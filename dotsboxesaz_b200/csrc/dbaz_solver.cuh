// dbaz_solver.cuh -- exact solver for boards of at most 32 real edges: a retrograde table of every position's value,
// and the per-state kernels that read it (move grading, a perfect-play evaluator for the search).
//
// Definitions (DESIGN.md §10):
//   E = 2LC + L + C real edges.  Compact edge index j = the j-th set bit of Board.real, in increasing action order;
//   M = the played edges as a uint32 compact mask.  Supported: E <= 32 (1x1..1x10, 2x2..2x6, 3x3, 3x4, transposes).
//   v(M) (int8) = the largest net number of boxes the player to move can still gain against best play, by the
//   full-game recurrence  v(full) = 0,  v(M) = max over free j of (c_j > 0 ? c_j + v(M|j) : -v(M|j)),
//   c_j = boxes edge j closes.
//   The mover's score lead d = (btc2[1-tp] - btc2[tp]) / 2 = LC - btc2[tp] - closed(M): a function of the eval-cache
//   key (edge set, btc2[tp]) alone.  Final margin = d + v(M); outcome = sign(d + v(M)) (the reference's result
//   convention, seen by the player to move).  The reference stops a game at a majority; sign is monotone and commutes
//   with max/min, so the outcome is the same.  Move margin of legal action a = d + (c > 0 ? c + v(M|a) : -v(M|a)); a
//   move is outcome-optimal if its sign equals the outcome, margin-optimal if it equals the final margin.
#pragma once
#include "dbaz_device.cuh"

namespace dbaz {

constexpr int SOLVER_MAX_EDGES = 32;
constexpr int SOLVER_MAX_BOXES = 16;
constexpr int8_t SOLVER_SENTINEL = -128;  // "not written" in the table; "illegal move" in move margins

// Compact geometry, built on the host from the engine's action table (k_build_act_tab) and passed by value.
struct SolverGeom {
    int E, LC, nboxes;
    uint8_t act[SOLVER_MAX_EDGES];        // action of compact edge j
    uint32_t ebox[SOLVER_MAX_EDGES][2];   // compact masks of the (up to) two boxes edge j borders; 0 = no box there
    uint32_t box[SOLVER_MAX_BOXES];       // compact mask of every box
};

// Binomial coefficients C(n, k), n, k <= 32 (C(32, 16) < 2^32): the combinatorial number system of k_solver_layer.
struct BinomTable {
    uint32_t c[SOLVER_MAX_EDGES + 1][SOLVER_MAX_EDGES + 1];
};
constexpr BinomTable make_binom() {
    BinomTable t{};
    for (int n = 0; n <= SOLVER_MAX_EDGES; ++n) {
        t.c[n][0] = 1;
        for (int k = 1; k <= n; ++k) t.c[n][k] = t.c[n - 1][k - 1] + (k <= n - 1 ? t.c[n - 1][k] : 0u);
    }
    return t;
}
__constant__ BinomTable c_binom = make_binom();
inline uint32_t c_binom_host(int n, int k) {
    static constexpr BinomTable t = make_binom();
    return t.c[n][k];
}

// The r-th k-subset of {0..E-1} in colex order (ascending masks): the largest c with C(c, i) <= r is element i.
__device__ __forceinline__ uint32_t colex_unrank(uint32_t r, int k, int E) {
    uint32_t m = 0;
    int c = E - 1;
    for (int i = k; i >= 1; --i) {
        while (c_binom.c[c][i] > r) --c;  // stops at c = i - 1 at the latest: C(i - 1, i) = 0
        m |= 1u << c;
        r -= c_binom.c[c][i];
        --c;
    }
    return m;
}

// boxes that compact edge j closes; `after` already holds j
__device__ __forceinline__ int solver_closes(const SolverGeom& g, uint32_t after, int j) {
    const uint32_t b0 = g.ebox[j][0], b1 = g.ebox[j][1];
    return ((b0 && (after & b0) == b0) ? 1 : 0) + ((b1 && (after & b1) == b1) ? 1 : 0);
}

__device__ __forceinline__ uint32_t solver_full(const SolverGeom& g) {
    return g.E == 32 ? 0xffffffffu : ((1u << g.E) - 1u);
}

// Entry r of layer k of a table over g.E edges: the r-th k-subset in colex order, so consecutive threads write increasing
// masks and their reads M | 1 << j of small j fall into shared sectors.  Layer k + 1 is complete (previous launch).
// One body for the full-board table (k_solver_layer) and the per-position tables of dbaz_endgame.cuh (k_deep_layer).
__device__ __forceinline__ void solver_layer_entry(const SolverGeom& g, int8_t* __restrict__ T, int k, uint32_t r) {
    const uint32_t M = colex_unrank(r, k, g.E);
    uint32_t fr = solver_full(g) & ~M;
    int best = SOLVER_SENTINEL;
    while (fr) {
        const int j = __ffs(fr) - 1;
        fr &= fr - 1;
        const uint32_t s = M | (1u << j);
        const int v = __ldg(reinterpret_cast<const signed char*>(T) + s);
        const int c = solver_closes(g, s, j);
        best = max(best, c ? c + v : -v);
    }
    T[M] = (int8_t)best;
}

// Layer k of the full-board table.
__global__ void __launch_bounds__(256) k_solver_layer(const __grid_constant__ SolverGeom g, int8_t* __restrict__ T, int k,
                                                      uint32_t count) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= count) return;
    solver_layer_entry(g, T, k, r);
}

// Number of sentinel bytes left in the table (16 bytes per thread and step; 2^E is a multiple of 16 for E >= 4).
__global__ void k_solver_check(const uint4* __restrict__ T, int64_t n16, unsigned long long* __restrict__ count) {
    unsigned int found = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n16; i += (int64_t)gridDim.x * blockDim.x) {
        const uint4 q = T[i];
        found += __popc(__vcmpeq4(q.x, 0x80808080u)) + __popc(__vcmpeq4(q.y, 0x80808080u)) +
                 __popc(__vcmpeq4(q.z, 0x80808080u)) + __popc(__vcmpeq4(q.w, 0x80808080u));
    }
    found /= 8;  // __vcmpeq4 sets all 8 bits of an equal byte
    for (int o = 16; o > 0; o >>= 1) found += __shfl_down_sync(0xffffffffu, found, o);
    if ((threadIdx.x & 31) == 0 && found) atomicAdd(count, (unsigned long long)found);
}

// What a warp knows of one state: compact mask, mover's lead, final margin.  Supported boards have A <= 44 actions,
// so every action lives in edge word 0.
struct SolverPos {
    uint32_t M;
    int d, final_margin;
};
__device__ __forceinline__ SolverPos solver_pos(const SolverGeom& g, const int8_t* __restrict__ T, const dbaz_state& s, int lane) {
    const bool bit = lane < g.E && ((s.edges[0] >> g.act[lane]) & 1ull);
    SolverPos p;
    p.M = __ballot_sync(0xffffffffu, bit);
    const bool closed = lane < g.nboxes && (p.M & g.box[lane]) == g.box[lane];
    const int n_closed = __popc(__ballot_sync(0xffffffffu, closed));
    const int mine2 = (s.to_play & 1) ? s.btc2[1] : s.btc2[0];
    p.d = g.LC - mine2 - n_closed;
    p.final_margin = p.d + (int)__ldg(reinterpret_cast<const signed char*>(T) + p.M);
    return p;
}

// move margin of action a (SOLVER_SENTINEL if a is not a free real edge)
__device__ __forceinline__ int solver_move_margin(const Board& b, const SolverGeom& g, const int8_t* __restrict__ T, const SolverPos& p,
                                                  int a) {
    if (a >= b.A || !((b.real[0] >> a) & 1ull)) return SOLVER_SENTINEL;
    const int j = __popcll(b.real[0] & ((1ull << a) - 1ull));
    if ((p.M >> j) & 1u) return SOLVER_SENTINEL;
    const uint32_t s = p.M | (1u << j);
    const int v = __ldg(reinterpret_cast<const signed char*>(T) + s);
    const int c = solver_closes(g, s, j);
    return p.d + (c ? c + v : -v);
}

__device__ __forceinline__ int sign_of(int x) { return (x > 0) - (x < 0); }

// One warp per state, lane = action: int8 move margins [n][A] and final margins [n].
__global__ void k_solver_moves(Board b, const __grid_constant__ SolverGeom g, const int8_t* __restrict__ T,
                               const dbaz_state* __restrict__ states, int8_t* __restrict__ move_margin,
                               int8_t* __restrict__ margin, int64_t n) {
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n) return;
    const dbaz_state s = states[w];
    const SolverPos p = solver_pos(g, T, s, lane);
    for (int a = lane; a < b.A; a += 32) move_margin[w * b.A + a] = (int8_t)solver_move_margin(b, g, T, p, a);
    if (lane == 0) margin[w] = (int8_t)p.final_margin;
}

// The perfect-play evaluator over the leaves the step kernel wrote: priors uniform over the outcome-optimal moves,
// value = outcome (mode 0) or final margin / (L C) (mode 1), both seen by the player to move at the leaf.
// A function of the eval-cache key: edge set and btc2[to_play].
__global__ void k_solver_eval(Board b, const __grid_constant__ SolverGeom g, const int8_t* __restrict__ T,
                              const dbaz_state* __restrict__ leaves, float* __restrict__ priors, float* __restrict__ values, int mode,
                              int64_t n) {
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n) return;
    const dbaz_state s = leaves[w];
    const SolverPos p = solver_pos(g, T, s, lane);
    const int o = sign_of(p.final_margin);
    constexpr int Q = 2;  // A <= 44 < 64
    bool opt[Q];
    int k = 0;
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const int mm = solver_move_margin(b, g, T, p, lane + 32 * q);
        opt[q] = mm != SOLVER_SENTINEL && sign_of(mm) == o;
        k += __popc(__ballot_sync(0xffffffffu, opt[q]));
    }
    const float u = k ? __fdiv_rn(1.0f, (float)k) : 0.0f;
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const int a = lane + 32 * q;
        if (a < b.A) priors[w * b.A + a] = opt[q] ? u : 0.0f;
    }
    if (lane == 0) values[w] = mode == 0 ? (float)o : __fdiv_rn((float)p.final_margin, (float)g.LC);
}

}  // namespace dbaz
