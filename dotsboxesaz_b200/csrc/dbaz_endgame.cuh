// dbaz_endgame.cuh -- exact endgame solver for every supported board (A <= 128): the retrograde of dbaz_solver.cuh run
// per position over its free edges only, in shared memory, and the per-state kernels that read it (move grading, an
// endgame-exact evaluator for the search).
//
// Definitions (DESIGN.md §11, extending §10):
//   F = the free real edges of a state, f = |F|.  Local edge i = the i-th set bit of Board.real & ~edges, in increasing
//   action order.  For a subset m of F a box closes when every one of its free edges is in m; boxes without a free edge
//   are closed already and take no part.  v_s(F) = 0, v_s(m) = max over i not in m of (c_i > 0 ? c_i + v_s(m|i) :
//   -v_s(m|i)), so v_s(0) = v(M) of §10 (M = the played edges).  Lead d, final margin d + v, outcome, move margins and
//   "outcome-optimal" / "margin-optimal" are those of §10.
//   A position is solvable when f <= max_free <= 16; every output of an unsolvable one is SOLVER_SENTINEL (-128) in the
//   move kernel and left untouched in the evaluator.
//
// Shape: one persistent kernel of ENDGAME_THREADS threads per CTA.  A CTA takes the rows blockIdx.x + gridDim.x * t
// (t = 0, 1, ...) ENDGAME_THREADS at a time: each thread classifies one row by f, then
//   f <= 10            one warp per position, a 1 KiB table per warp, __syncwarp between popcount layers;
//   11 <= f <= 16      the whole CTA per position, a 2^f-byte table, __syncthreads between popcount layers.
// Layer k of an f-edge table is the k-subsets of f bits in increasing order, read from a table of every such ordering
// (endgame_order_host, uploaded once per engine), so a thread reads its mask instead of unranking it.
// Where the rows come from is a template parameter (Rows): a contiguous state array here (StateRows), the roots of the
// self-play trees in dbaz_selfplay.cuh.  A row the source does not qualify is classified unsolvable without being read.
#pragma once
#include "dbaz_solver.cuh"

namespace dbaz {

constexpr int ENDGAME_MAX_FREE = 16;
constexpr int ENDGAME_WARP_MAX_FREE = 10;  // positions with f <= 10 are solved by one warp
constexpr int ENDGAME_THREADS = 512;
constexpr int ENDGAME_WARPS = ENDGAME_THREADS / 32;
constexpr int ENDGAME_ORDER_ENTRIES = (2 << ENDGAME_MAX_FREE) - 1;  // 2^0 + 2^1 + ... + 2^16 masks

// Dynamic shared memory of a launch: the CTA tier's 2^max_free-byte table or the warp tier's 16 x 1 KiB, the larger.
inline int endgame_smem_bytes(int max_free) {
    const int cta = 1 << max_free, warps = ENDGAME_WARPS << ENDGAME_WARP_MAX_FREE;
    return cta > warps ? cta : warps;
}

// Entry (2^f - 1) + r of `out` is the r-th mask of f bits in order of (popcount, value): layer k of an f-edge table
// starts at sum over j < k of C(f, j).
inline void endgame_order_host(uint16_t* out) {
    for (int f = 0; f <= ENDGAME_MAX_FREE; ++f) {
        uint32_t pos[ENDGAME_MAX_FREE + 1];
        uint32_t at = (1u << f) - 1u;
        for (int k = 0; k <= f; ++k) { pos[k] = at; at += c_binom_host(f, k); }
        for (uint32_t m = 0; m < (1u << f); ++m) out[pos[__builtin_popcount(m)]++] = (uint16_t)m;
    }
}

// What a warp knows of one row: its free edges, their number and the mover's lead.
struct EndgameRow {
    uint64_t F0, F1;
    int f, d;
};

__device__ __forceinline__ int endgame_f(const Board& b, const dbaz_state& s) {
    return __popcll(b.real[0] & ~s.edges[0]) + __popcll(b.real[1] & ~s.edges[1]);
}

// local index of free action a: the free edges below it
__device__ __forceinline__ int endgame_rank(uint64_t F0, uint64_t F1, int a) {
    return a < 64 ? __popcll(F0 & ((1ull << a) - 1ull)) : __popcll(F0) + __popcll(F1 & ((1ull << (a - 64)) - 1ull));
}

// local mask of the free edges of an action-space box mask (0 for no box)
__device__ __forceinline__ uint32_t endgame_local(uint64_t F0, uint64_t F1, uint64_t w0, uint64_t w1) {
    uint32_t m = 0;
    for (w0 &= F0; w0; w0 &= w0 - 1ull) m |= 1u << endgame_rank(F0, F1, __ffsll((long long)w0) - 1);
    for (w1 &= F1; w1; w1 &= w1 - 1ull) m |= 1u << endgame_rank(F0, F1, 64 + __ffsll((long long)w1) - 1);
    return m;
}

// action of local edge i (f0 = free edges in word 0)
__device__ __forceinline__ int endgame_action(uint64_t F0, uint64_t F1, int f0, int i) {
    return i < f0 ? nth_set_bit(F0, i) : 64 + nth_set_bit(F1, i - f0);
}

// local mask of box k (0 or 1, from act_tab) of action a: its free edges (0 for no box)
__device__ __forceinline__ uint32_t endgame_edge_box(const uint4* __restrict__ act_tab, uint64_t F0, uint64_t F1, int a, int k) {
    const uint4 q = __ldg(act_tab + 2 * a + k);
    return endgame_local(F0, F1, (uint64_t)q.x | ((uint64_t)q.y << 32), (uint64_t)q.z | ((uint64_t)q.w << 32));
}

// Whole warp: the mover's lead d = LC - btc2[to_play] - closed boxes; box (l, c) is the second box of its top edge
// l * cols + c.
__device__ __forceinline__ int endgame_lead(const Board& b, const uint4* __restrict__ act_tab, const dbaz_state& s, int lane) {
    int closed = 0;
    for (int x = lane; x < b.nboxes; x += 32) {
        const int l = x / b.C, c = x - l * b.C;
        const uint4 q = __ldg(act_tab + 2 * (l * b.cols + c) + 1);
        const uint64_t w0 = (uint64_t)q.x | ((uint64_t)q.y << 32), w1 = (uint64_t)q.z | ((uint64_t)q.w << 32);
        closed += ((s.edges[0] & w0) == w0 && (s.edges[1] & w1) == w1) ? 1 : 0;
    }
    closed = __reduce_add_sync(0xffffffffu, closed);
    const int mine2 = (s.to_play & 1) ? s.btc2[1] : s.btc2[0];
    return b.nboxes - mine2 - closed;
}

// Whole warp: the row's free edges and lead, and geo[i] = the local masks of the (up to) two boxes local edge i borders
// (low / high 16 bits) for i < f <= 16.
__device__ __forceinline__ EndgameRow endgame_row(const Board& b, const uint4* __restrict__ act_tab, const dbaz_state& s,
                                                  uint32_t* geo, int lane) {
    EndgameRow p;
    p.F0 = b.real[0] & ~s.edges[0];
    p.F1 = b.real[1] & ~s.edges[1];
    const int f0 = __popcll(p.F0);
    p.f = f0 + __popcll(p.F1);
    if (lane < p.f && lane < ENDGAME_MAX_FREE) {
        const int a = endgame_action(p.F0, p.F1, f0, lane);
        uint32_t eb = 0;
#pragma unroll
        for (int k = 0; k < 2; ++k) eb |= endgame_edge_box(act_tab, p.F0, p.F1, a, k) << (16 * k);
        geo[lane] = eb;
    }
    p.d = endgame_lead(b, act_tab, s, lane);
    return p;
}

template <int G>
__device__ __forceinline__ void endgame_sync() {
    if (G == 32) __syncwarp();
    else __syncthreads();
}

// G threads (a warp or the CTA; tid in [0, G)) fill T[0 .. 2^f) with v_s, one popcount layer at a time.  All threads of a
// layer have f - k free bits, so the successor loop has the same trip count across the group.
template <int G>
__device__ __forceinline__ void endgame_table(int8_t* T, const uint32_t* geo, int f, int tid, const uint16_t* __restrict__ order) {
    const uint32_t full = (1u << f) - 1u;
    if (tid == 0) T[full] = 0;
    endgame_sync<G>();
    const uint16_t* ord = order + full;  // the masks of f bits start at 2^f - 1
    uint32_t off = full;                 // start of layer k: layer f (the full set) is the last entry
    for (int k = f - 1; k >= 0; --k) {
        const uint32_t cnt = c_binom.c[f][k];
        off -= cnt;
        for (uint32_t r = tid; r < cnt; r += G) {
            const uint32_t m = __ldg(ord + off + r);
            int best = SOLVER_SENTINEL;
            for (uint32_t fr = full & ~m; fr; fr &= fr - 1u) {
                const int i = __ffs(fr) - 1;
                const uint32_t s = m | (1u << i);
                const int v = T[s];
                const uint32_t eb = geo[i], b0 = eb & 0xffffu, b1 = eb >> 16;
                const int c = ((b0 && (s & b0) == b0) ? 1 : 0) + ((b1 && (s & b1) == b1) ? 1 : 0);
                best = max(best, c ? c + v : -v);
            }
            T[m] = (int8_t)best;
        }
        endgame_sync<G>();
    }
}

// move margin of action a from a filled table (SOLVER_SENTINEL if a is not a free edge)
__device__ __forceinline__ int endgame_move_margin(const Board& b, const EndgameRow& p, const int8_t* T, const uint32_t* geo, int a) {
    if (a >= b.A) return SOLVER_SENTINEL;
    const bool free = a < 64 ? ((p.F0 >> a) & 1ull) : ((p.F1 >> (a - 64)) & 1ull);
    if (!free) return SOLVER_SENTINEL;
    const int i = endgame_rank(p.F0, p.F1, a);
    const uint32_t bit = 1u << i, eb = geo[i];
    const int c = ((eb & 0xffffu) == bit ? 1 : 0) + ((eb >> 16) == bit ? 1 : 0);  // a box closes iff i is its last free edge
    const int v = T[bit];
    return p.d + (c ? c + v : -v);
}

// k_endgame_moves' output: int8 move margins [n][A] and final margins [n], as k_solver_moves
struct EndgameMovesOut {
    int8_t* move_margin;
    int8_t* margin;
    static constexpr bool kUnsolvable = true;
    __device__ __forceinline__ void unsolvable(const Board& b, int64_t w, int lane) const {
        for (int a = lane; a < b.A; a += 32) move_margin[w * b.A + a] = SOLVER_SENTINEL;
        if (lane == 0) margin[w] = SOLVER_SENTINEL;
    }
    __device__ __forceinline__ void solved(const Board& b, const EndgameRow& p, const int8_t* T, const uint32_t* geo, int64_t w,
                                           int lane) const {
        for (int a = lane; a < b.A; a += 32) move_margin[w * b.A + a] = (int8_t)endgame_move_margin(b, p, T, geo, a);
        if (lane == 0) margin[w] = (int8_t)(p.d + T[0]);
    }
};

// k_endgame_eval's output, as k_solver_eval: priors uniform over the outcome-optimal moves (unless keep_priors), value =
// outcome (mode 0) or final margin / (L C) (mode 1).  Unsolvable rows keep what the inner evaluator wrote.
struct EndgameEvalOut {
    float* priors;
    float* values;
    int mode, keep_priors;
    static constexpr bool kUnsolvable = false;
    __device__ __forceinline__ void unsolvable(const Board&, int64_t, int) const {}
    __device__ __forceinline__ void solved(const Board& b, const EndgameRow& p, const int8_t* T, const uint32_t* geo, int64_t w,
                                           int lane) const {
        const int final_margin = p.d + T[0];
        const int o = sign_of(final_margin);
        if (!keep_priors) {
            constexpr int Q = DBAZ_MAX_ACTIONS / 32;
            bool opt[Q];
            int k = 0;
#pragma unroll
            for (int q = 0; q < Q; ++q) {
                const int mm = endgame_move_margin(b, p, T, geo, lane + 32 * q);
                opt[q] = mm != SOLVER_SENTINEL && sign_of(mm) == o;
                k += __popc(__ballot_sync(0xffffffffu, opt[q]));
            }
            const float u = k ? __fdiv_rn(1.0f, (float)k) : 0.0f;
#pragma unroll
            for (int q = 0; q < Q; ++q) {
                const int a = lane + 32 * q;
                if (a < b.A) priors[w * b.A + a] = opt[q] ? u : 0.0f;
            }
        }
        if (lane == 0) values[w] = mode == 0 ? (float)o : __fdiv_rn((float)final_margin, (float)b.nboxes);
    }
};

// Row source of k_endgame_moves / k_endgame_eval: state w of a contiguous array, every row qualifies.
struct StateRows {
    const dbaz_state* __restrict__ states;
    __device__ __forceinline__ bool qualifies(int64_t) const { return true; }
    __device__ __forceinline__ dbaz_state state(int64_t w) const { return states[w]; }
};

template <class Rows, class Out>
__device__ __forceinline__ void endgame_rows(const Board& b, const uint4* __restrict__ act_tab, const uint16_t* __restrict__ order,
                                             const Rows& rows, const Out& out, int max_free, int64_t n) {
    extern __shared__ __align__(16) int8_t eg_table[];  // endgame_smem_bytes(max_free)
    __shared__ uint32_t geo[ENDGAME_WARPS][ENDGAME_MAX_FREE];
    __shared__ uint16_t list[3][ENDGAME_THREADS];  // rows of this pass for the warp tier, the CTA tier, unsolvable
    __shared__ int count[3];
    __shared__ int cta_f;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int warp_max = min(max_free, ENDGAME_WARP_MAX_FREE);
    const int64_t stride = gridDim.x;
    for (int64_t first = blockIdx.x; first < n; first += stride * ENDGAME_THREADS) {
        if (tid < 3) count[tid] = 0;
        __syncthreads();
        const int64_t w = first + stride * tid;
        if (w < n) {
            const int f = rows.qualifies(w) ? endgame_f(b, rows.state(w)) : ENDGAME_MAX_FREE + 1;
            const int tier = f <= warp_max ? 0 : f <= max_free ? 1 : 2;
            list[tier][atomicAdd(&count[tier], 1)] = (uint16_t)tid;
        }
        __syncthreads();
        if (Out::kUnsolvable)
            for (int j = warp; j < count[2]; j += ENDGAME_WARPS) out.unsolvable(b, first + stride * list[2][j], lane);
        int8_t* Tw = eg_table + (warp << ENDGAME_WARP_MAX_FREE);
        for (int j = warp; j < count[0]; j += ENDGAME_WARPS) {
            const int64_t row = first + stride * list[0][j];
            const dbaz_state s = rows.state(row);
            const EndgameRow p = endgame_row(b, act_tab, s, geo[warp], lane);
            __syncwarp();
            endgame_table<32>(Tw, geo[warp], p.f, lane, order);
            out.solved(b, p, Tw, geo[warp], row, lane);
            __syncwarp();  // the next row rewrites geo and the table
        }
        __syncthreads();
        for (int j = 0; j < count[1]; ++j) {
            const int64_t row = first + stride * list[1][j];
            EndgameRow p;
            if (warp == 0) {
                const dbaz_state s = rows.state(row);
                p = endgame_row(b, act_tab, s, geo[0], lane);
                if (lane == 0) cta_f = p.f;
            }
            __syncthreads();
            endgame_table<ENDGAME_THREADS>(eg_table, geo[0], cta_f, tid, order);
            if (warp == 0) out.solved(b, p, eg_table, geo[0], row, lane);
            // the other warps wait for warp 0's next geometry at the barrier above before touching the table again
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(ENDGAME_THREADS, 3) k_endgame_moves(Board b, const uint4* __restrict__ act_tab,
                                                                  const uint16_t* __restrict__ order, const dbaz_state* __restrict__ states,
                                                                  EndgameMovesOut out, int max_free, int64_t n) {
    endgame_rows(b, act_tab, order, StateRows{states}, out, max_free, n);
}

__global__ void __launch_bounds__(ENDGAME_THREADS, 3) k_endgame_eval(Board b, const uint4* __restrict__ act_tab,
                                                                 const uint16_t* __restrict__ order, const dbaz_state* __restrict__ leaves,
                                                                 EndgameEvalOut out, int max_free, int64_t n) {
    endgame_rows(b, act_tab, order, StateRows{leaves}, out, max_free, n);
}

// ---- deep tier (DESIGN.md §13): positions with 17 <= f <= 32 free edges, one 2^f-byte table per position in device
// memory, solved by the layer body of k_solver_layer over local edges.  A pass of P positions, all with the same f, uses
// a caller-owned workspace: table p at ws + p 2^f, then geometry slot p at ws + P 2^f + p ENDGAME_DEEP_GEOM_BYTES.
constexpr int ENDGAME_DEEP_MIN_FREE = ENDGAME_MAX_FREE + 1;
constexpr int ENDGAME_DEEP_MAX_FREE = SOLVER_MAX_EDGES;
constexpr int ENDGAME_DEEP_GEOM_BYTES = 512;
constexpr int ENDGAME_DEEP_MAX_PASS = 65535;  // positions per pass: gridDim.y of k_deep_layer

// One position's geometry in SolverGeom's shape: E = f and ebox = the local box masks of its free edges (act, box, LC and
// nboxes are not used), plus the mover's lead.
struct DeepGeom {
    SolverGeom g;
    int d;
};
static_assert(sizeof(DeepGeom) <= ENDGAME_DEEP_GEOM_BYTES, "a deep geometry slot holds a DeepGeom");

__device__ __forceinline__ DeepGeom* deep_geom(int8_t* ws, int f, int P, int p) {
    return reinterpret_cast<DeepGeom*>(ws + ((int64_t)P << f) + (int64_t)p * ENDGAME_DEEP_GEOM_BYTES);
}

// One warp per position of the pass: its geometry and the full-set entry T_p[2^f - 1] = 0 (the rest of the tables is the
// sentinel).  A state whose f is not the launch's is counted in *mismatch and gets an empty geometry.
__global__ void k_deep_geom(Board b, const uint4* __restrict__ act_tab, const dbaz_state* __restrict__ states, int8_t* ws, int f, int P,
                            unsigned long long* __restrict__ mismatch) {
    const int p = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= P) return;
    const dbaz_state s = states[p];
    const uint64_t F0 = b.real[0] & ~s.edges[0], F1 = b.real[1] & ~s.edges[1];
    const int f0 = __popcll(F0);
    const bool ok = f0 + __popcll(F1) == f;
    DeepGeom* G = deep_geom(ws, f, P, p);
    uint32_t eb[2] = {0u, 0u};
    if (ok && lane < f) {
        const int a = endgame_action(F0, F1, f0, lane);
        eb[0] = endgame_edge_box(act_tab, F0, F1, a, 0);
        eb[1] = endgame_edge_box(act_tab, F0, F1, a, 1);
    }
    G->g.ebox[lane][0] = eb[0];
    G->g.ebox[lane][1] = eb[1];
    const int d = endgame_lead(b, act_tab, s, lane);
    if (lane == 0) {
        G->g.E = f;
        G->d = d;
        ws[((int64_t)p << f) + (((int64_t)1 << f) - 1)] = 0;
        if (!ok) atomicAdd(mismatch, 1ull);
    }
}

// Layer k of every table of the pass: blockIdx.y = position, blockIdx.x * 256 + threadIdx.x = entry of the layer.
__global__ void __launch_bounds__(256) k_deep_layer(int8_t* ws, int f, int P, int k, uint32_t count) {
    __shared__ SolverGeom g;
    const int p = blockIdx.y;
    const DeepGeom* G = deep_geom(ws, f, P, p);
    if (threadIdx.x < 2 * SOLVER_MAX_EDGES) g.ebox[threadIdx.x >> 1][threadIdx.x & 1] = G->g.ebox[threadIdx.x >> 1][threadIdx.x & 1];
    if (threadIdx.x == 0) g.E = f;
    __syncthreads();
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= count) return;
    solver_layer_entry(g, ws + ((int64_t)p << f), k, r);
}

// One warp per position of the pass, from its filled table: move margins [P][A] and final margins [P] as k_endgame_moves.
// A box closes iff local edge i is its last free edge (ebox == 1 << i).
__global__ void k_deep_moves(Board b, const dbaz_state* __restrict__ states, int8_t* ws, int f, int P, int8_t* __restrict__ move_margin,
                             int8_t* __restrict__ margin) {
    const int p = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= P) return;
    const dbaz_state s = states[p];
    const uint64_t F0 = b.real[0] & ~s.edges[0], F1 = b.real[1] & ~s.edges[1];
    const DeepGeom* G = deep_geom(ws, f, P, p);
    const int8_t* T = ws + ((int64_t)p << f);
    const int d = G->d;
    for (int a = lane; a < b.A; a += 32) {
        int mm = SOLVER_SENTINEL;
        if (a < 64 ? ((F0 >> a) & 1ull) : ((F1 >> (a - 64)) & 1ull)) {
            const int i = endgame_rank(F0, F1, a);
            const uint32_t bit = 1u << i;
            const int c = (G->g.ebox[i][0] == bit ? 1 : 0) + (G->g.ebox[i][1] == bit ? 1 : 0);
            const int v = T[bit];
            mm = d + (c ? c + v : -v);
        }
        move_margin[(int64_t)p * b.A + a] = (int8_t)mm;
    }
    if (lane == 0) margin[p] = (int8_t)(d + T[0]);
}

}  // namespace dbaz
