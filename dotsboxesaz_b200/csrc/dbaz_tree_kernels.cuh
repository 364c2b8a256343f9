// dbaz_tree_kernels.cuh -- the per-simulation hot path: PUCT select, lazy child creation,
// feature gather, expand, backup, root-prior mix, re-root with in-place subtree compaction.
//
// One warp owns one tree (one game) and runs its simulations in the reference's order, so no
// atomics are needed and visit counts are bit-identical to the reference's UCT_search:
// with max_pending_evals = 1 strictly one simulation after the other; with max_pending_evals = K
// in the waves the reference's event loop produces (K select_leaf()s leaving their virtual loss
// behind, a terminal leaf backed up on the spot, then the K expand/backup pairs in the same order;
// mcts.py:228-242).  Parallelism comes from the thousands of trees.
//
// What a launch of k_search_step does for one tree (max_pending_evals = 1, search_step_seq): back up the leaf the
// evaluator answered, then run simulations back to back for as long as they need no evaluator -- terminal leaves and
// leaves found in the eval cache (the reference's LRU of net outputs, utils/proxies.py:35-43) finish on the spot --
// until a leaf needs the net: it goes to the next free row of the evaluator's batch (or waits a wave if the batch is
// full).  The selection loop stores nothing but lazily created children; path and statistics stay in registers.
//
// HBM layout per tree t (arena[t] = max_nodes fixed-stride nodes):
//   node i : [ dbaz_state header 32 B | Child rec[A] 16 B each ]      stride = 32 + 16*A
// A node's own N/W live in its parent's Child record (as in mcts.py:67-89); the root's live
// in TreeRec (TreeRoot, mcts.py:21-36).  Node 0 is always the root (re-rooting compacts the
// kept subtree to the front of the arena), so Child.child == 0 means "not created".
//
// Reference behaviour restated (paths relative to the reference root):
//   mcts.py:91-103   children_ucb_score / best_child  -> ucb_score() + warp_argmax() inside tree_select()
//   mcts.py:105-114  select_leaf                      -> tree_select()
//   mcts.py:116-132  expand / backup                  -> tree_expand_backup()
//   mcts.py:184-199  _search                          -> search_step_seq() / search_step_waves() in k_search_step
//   utils/proxies.py:35-43  LRU of net outputs        -> cache_lookup() / cache_insert()
//   mcts.py:205-229  UCT_search head (root prior mix) -> root_prior_mix()
//   mcts.py:163-180  init_mcts_tree                   -> k_advance_roots
#pragma once
#include "dbaz_device.cuh"

namespace dbaz {

enum : uint32_t {
    TF_PRIOR_SET = 1,      // root_prior[t] holds this root's child_priors (set by a UCT_search head)
    TF_PRIOR_F64 = 2,      // ... and they were produced by float64 arithmetic
    TF_PREP_PENDING = 4,   // root was unexpanded at begin(): mix priors after its first backup
    TF_ERR_POOL = 8,       // node pool exhausted
    TF_ERR_MOVE = 16,      // advance_roots with an illegal move
    TF_FIRST_WAVE = 32,    // next wave is the first of this UCT_search: min(max_pending_evals, A) wide (mcts.py:228-229)
};

struct __align__(64) TreeRec {
    int32_t n_nodes;
    int32_t root_N;       // TreeRoot.child_number_visits[None]
    float root_W;         // TreeRoot.child_total_value[None] (float32 in effect)
    int32_t sims_left;
    int32_t n_pending;    // simulations selected and waiting for their evaluation (<= max_pending)
    int32_t row;          // compact mode: row of the evaluator's batch that holds this tree's pending leaf
    uint32_t flags;
    int32_t max_deepness;
    int32_t deepness_correction;
    int32_t terminal_count;
    int32_t tree_size;
    int32_t total_term;   // terminal leaves since reset (instrumentation)
    uint32_t total_sims;  // simulations since reset (instrumentation)
    uint32_t cache_hits;  // ... of which the evaluation came out of the eval cache
    unsigned long long total_path;
};
static_assert(sizeof(TreeRec) == 64, "TreeRec must be 64 bytes");

// the fields a wave carries in registers (first 32 bytes of TreeRec); the statistics stay in memory
struct TreeHot {
    int32_t n_nodes, root_N;
    float root_W;
    int32_t sims_left, n_pending, row;
    uint32_t flags;
};
__device__ __forceinline__ TreeHot load_hot(const TreeRec* G) {
    const uint4 a = reinterpret_cast<const uint4*>(G)[0];
    const uint4 b = reinterpret_cast<const uint4*>(G)[1];
    TreeHot T;
    T.n_nodes = (int)a.x; T.root_N = (int)a.y; T.root_W = __uint_as_float(a.z); T.sims_left = (int)a.w;
    T.n_pending = (int)b.x; T.row = (int)b.y; T.flags = b.z;
    return T;
}
__device__ __forceinline__ void store_hot(TreeRec* G, const TreeHot& T) {
    reinterpret_cast<uint4*>(G)[0] = make_uint4((uint32_t)T.n_nodes, (uint32_t)T.root_N, __float_as_uint(T.root_W), (uint32_t)T.sims_left);
    reinterpret_cast<uint2*>(G)[2] = make_uint2((uint32_t)T.n_pending, (uint32_t)T.row);
    G->flags = T.flags;
}

constexpr int PATH_CAP = 128;               // >= number of real edges + 1
constexpr uint32_t PATH_ROOT = 0x7fffff00u; // parent field of the root's path element

struct TreeArgs {
    char* arena;          // n_trees * max_nodes * stride bytes
    TreeRec* trees;
    double* root_prior;   // [n_trees][A]
    uint32_t* path;       // [max_pending][n_trees][PATH_CAP]
    uint2* path_wn;       // [n_trees][PATH_CAP]: {W, N} of each path node's own record as the selection saw them (sequential mode)
    const double2* lut;   // {c0(N) = log((N + base + 1)/base) + cpuct, sqrt(N)}, host libm
    const uint4* act_tab; // [A][2]: the two box masks each action borders (built once per engine)
    uint4* pend;          // [max_pending][n_trees][3]: pending leaf {header copy (2 x 16 B), node index, path length}
    int max_pending;      // lanes of in-flight simulations per tree; row of lane k of tree t = k * n_trees + t
    int lut_size;
    int n_trees;
    int max_nodes;
    int stride;           // node stride in bytes
    double cpuct, cpuct_base;
    // evaluation cache (utils/proxies.py:23-26,35-43): direct-mapped table of cache_mask + 1 entries of A 16-byte cells
    // {p_a, key[3]}; the value rides in the cell of padding action `cache_vcell`.  nullptr = disabled.
    uint4* cache;
    uint32_t cache_mask;
    int cache_vcell;
    // table epoch (device memory: the captured step kernels must see a later clear): part of every key, so bumping it
    // empties the table without touching its gigabytes (dbaz_cache_clear)
    const uint32_t* cache_epoch;
    // lock-step bookkeeping, self-resetting (the last CTA of a launch publishes and zeroes it):
    // ctr[0..1] one 64-bit word {bits 40+: rows asked for, 20-39: trees still busy, 0-19: warps done} | ctr[4] rows asked for by the last launch,
    // ctr[5] busy trees after it, ctr[6] largest ctr[4] since the host last read it, ctr[7] largest node pool use seen by a re-root
    int* ctr;
    int compact;          // 1: a tree's pending leaf goes to row atomicAdd(ctr[0]) instead of row == tree (pending == 1 only)
    int max_inline;       // > 0: at most this many simulations per tree and launch may finish without the net
    int chain_clk;        // > 0: ... and none is started once the tree has spent this many SM clocks in the launch
    int batch_rows;       // compact mode: rows the evaluator of this launch will run; a leaf beyond them waits a wave
};

__device__ __forceinline__ char* node_ptr(const TreeArgs& ta, int t, int i) {
    return ta.arena + ((int64_t)t * ta.max_nodes + i) * (int64_t)ta.stride;
}
__device__ __forceinline__ dbaz_state load_hdr(const char* np) {
    // 32-byte header as two 16-byte loads; every lane reads the same address (broadcast)
    union { dbaz_state s; int4 v[2]; } u;
    const int4* p = reinterpret_cast<const int4*>(np);
    u.v[0] = p[0]; u.v[1] = p[1];
    return u.s;
}
__device__ __forceinline__ void store_hdr(char* np, const dbaz_state& s) {
    union { dbaz_state s; int4 v[2]; } u;
    u.s = s;
    int4* p = reinterpret_cast<int4*>(np);
    p[0] = u.v[0]; p[1] = u.v[1];
}
__device__ __forceinline__ Child* node_children(char* np) { return reinterpret_cast<Child*>(np + 32); }

// The 32-byte node header unpacked into registers (same byte layout as dbaz_state; going through the
// struct would spill it to local memory).
struct Hdr {
    uint64_t e0, e1;
    int btc0, btc1, to_play, just_played, flags, depth, parent, parent_action, result;
};
__device__ __forceinline__ Hdr unpack_hdr(const uint4& a, const uint4& b) {
    Hdr h;
    h.e0 = (uint64_t)a.x | ((uint64_t)a.y << 32);
    h.e1 = (uint64_t)a.z | ((uint64_t)a.w << 32);
    h.btc0 = (int)(int16_t)(b.x & 0xffffu); h.btc1 = (int)(int16_t)(b.x >> 16);
    h.to_play = b.y & 0xffu; h.just_played = (int)(int8_t)((b.y >> 8) & 0xffu);
    h.flags = (b.y >> 16) & 0xffu; h.depth = (b.y >> 24) & 0xffu;
    h.parent = (int)b.z;
    h.parent_action = (int)(int16_t)(b.w & 0xffffu); h.result = (int)(int16_t)(b.w >> 16);
    return h;
}
__device__ __forceinline__ void pack_hdr(const Hdr& h, uint4& a, uint4& b) {
    a.x = (uint32_t)h.e0; a.y = (uint32_t)(h.e0 >> 32); a.z = (uint32_t)h.e1; a.w = (uint32_t)(h.e1 >> 32);
    b.x = ((uint32_t)h.btc0 & 0xffffu) | ((uint32_t)h.btc1 << 16);
    b.y = ((uint32_t)h.to_play & 0xffu) | (((uint32_t)h.just_played & 0xffu) << 8) | (((uint32_t)h.flags & 0xffu) << 16) |
          (((uint32_t)h.depth & 0xffu) << 24);
    b.z = (uint32_t)h.parent;
    b.w = ((uint32_t)h.parent_action & 0xffffu) | ((uint32_t)h.result << 16);
}
__device__ __forceinline__ Hdr load_hdr_regs(const char* np) {
    const uint4* p = reinterpret_cast<const uint4*>(np);
    uint4 a = p[0], b = p[1];
    return unpack_hdr(a, b);
}
__device__ __forceinline__ void store_hdr_regs(char* np, const Hdr& h) {
    uint4 a, b;
    pack_hdr(h, a, b);
    uint4* p = reinterpret_cast<uint4*>(np);
    p[0] = a; p[1] = b;
}
__device__ __forceinline__ int hdr_result(const Hdr& h) {  // dots_boxes_game.py:51-59
    const int mine = h.to_play ? h.btc1 : h.btc0, other = h.to_play ? h.btc0 : h.btc1;
    if (h.btc0 == 0 && h.btc1 == 0) return 0;
    if (mine < 0) return 1;
    if (other < 0) return -1;
    return DBAZ_RESULT_NONE;
}
template <int NW>
__device__ __forceinline__ Mask<NW> hdr_edges(const Hdr& h) {
    Mask<NW> m;
    m.w[0] = h.e0;
    if (NW == 2) m.w[NW - 1] = h.e1;
    return m;
}

// {c0(N), sqrt(N)} of mcts.py:92-94 for a node with N own visits: one 16-byte load from a table the host built with
// libm (the functions CPython's math.log / math.sqrt call), issued together with the node's loads, instead of a
// float64 log + sqrt instruction chain behind them.
__device__ __forceinline__ double2 puct_consts(const TreeArgs& ta, int N) {
    if (N < ta.lut_size) return ta.lut[N];
    // beyond the host table: device log (<= 1 ulp from libm; documented in DESIGN.md), IEEE sqrt
    double2 r;
    r.x = __dadd_rn(log(__ddiv_rn(__dadd_rn(__dadd_rn((double)N, ta.cpuct_base), 1.0), ta.cpuct_base)), ta.cpuct);
    r.y = __dsqrt_rn((double)N);
    return r;
}

// Per-lane constants of the lane -> action mapping (action = lane + 32*k): own bit and the two
// boxes each action borders.  Computed once per kernel, reused at every level of every tree.
template <int APL, int NW>
struct LaneActions {
    Mask<NW> box[APL][2];
    bool real[APL];
    __device__ __forceinline__ void load(const Board& b, const uint4* __restrict__ tab, int lane) {
#pragma unroll
        for (int k = 0; k < APL; ++k) {
            const int a = lane + 32 * k;
            real[k] = a < b.A && ((b.real[a >> 6] >> (a & 63)) & 1ull);
            uint4 m0 = make_uint4(0, 0, 0, 0), m1 = m0;
            if (a < b.A) { m0 = tab[2 * a]; m1 = tab[2 * a + 1]; }
            box[k][0].w[0] = (uint64_t)m0.x | ((uint64_t)m0.y << 32);
            box[k][1].w[0] = (uint64_t)m1.x | ((uint64_t)m1.y << 32);
            if (NW == 2) {
                box[k][0].w[NW - 1] = (uint64_t)m0.z | ((uint64_t)m0.w << 32);
                box[k][1].w[NW - 1] = (uint64_t)m1.z | ((uint64_t)m1.w << 32);
            }
        }
    }
    // boxes closed by action k of this lane on edges e (before the move)
    __device__ __forceinline__ int closes(int k, const Mask<NW>& e, int a) const {
        Mask<NW> ea = e;
        mask_set(ea, a);
        return closed_count<NW>(ea, box[k]);
    }
};

// one thread per action: the two box masks the action borders, in play_'s test order
__global__ void k_build_act_tab(Board b, uint4* __restrict__ tab) {
    int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= b.A) return;
    Mask<2> box[2];
    int lc[2][2];
    action_boxes<2>(b, a, box, lc);
    for (int j = 0; j < 2; ++j)
        tab[2 * a + j] = make_uint4((uint32_t)box[j].w[0], (uint32_t)(box[j].w[0] >> 32), (uint32_t)box[j].w[1], (uint32_t)(box[j].w[1] >> 32));
}

// One PUCT level (mcts.py:91-103), float64 with every operation individually rounded (no FMA):
//   pb_c = c0(N) * (sqrt(N) / (n_i + 1)); score_i = pb_c * prior_i + (W_i / (1 + n_i)) * sign_i
//   argmax over legal actions, lowest action id wins ties (np.argmax).
template <int APL, int NW>
__device__ __forceinline__ double ucb_score(double c0, double sq, const Child& c, double prior, int sign) {
    double pb = __dmul_rn(c0, __ddiv_rn(sq, (double)(c.N + 1)));
    double ps = __dmul_rn(pb, prior);
    double vs = __dmul_rn(__ddiv_rn((double)c.W, (double)(1 + c.N)), (double)sign);
    return __dadd_rn(ps, vs);
}

// Root prior mix, head of UCT_search (mcts.py:213-226).  Warp-cooperative; `sh` is a per-warp
// shared scratch of A doubles.  noise == nullptr <=> alpha <= 0.
template <int APL, int NW>
__device__ __forceinline__ void root_prior_mix(const Board& b, const TreeArgs& ta, int t, TreeHot& T, const dbaz_state& rh,
                                               const double* noise, double coeff, double* sh, int lane) {
    const int A = b.A;
    double* rp = ta.root_prior + (int64_t)t * A;
    bool f64;
    // source: the root's current child_priors
    if (T.flags & TF_PRIOR_SET) {
        f64 = T.flags & TF_PRIOR_F64;
        for (int a = lane; a < A; a += 32) sh[a] = rp[a];
    } else if ((rh.flags & NF_EXPANDED) && !(rh.flags & NF_TERMINAL)) {
        f64 = false;
        const Child* ch = node_children(node_ptr(ta, t, 0));
        for (int a = lane; a < A; a += 32) sh[a] = (double)ch[a].prior;
    } else {  // terminal root: np.zeros(A), float64
        f64 = true;
        for (int a = lane; a < A; a += 32) sh[a] = 0.0;
    }
    __syncwarp();
    double probs[APL];
    bool probs_f64;
    if (f64) {
        double s = np_sum<double>(sh, A);
        probs_f64 = true;
#pragma unroll
        for (int k = 0; k < APL; ++k) {
            int a = lane + 32 * k;
            probs[k] = (a < A) ? (s != 0.0 ? __ddiv_rn(sh[a], s) : 0.0) : 0.0;
        }
    } else {
        // float32 arithmetic on float32 data: stage as floats in the same scratch
        float* shf = reinterpret_cast<float*>(sh);
        float mine[APL];
#pragma unroll
        for (int k = 0; k < APL; ++k) { int a = lane + 32 * k; mine[k] = a < A ? (float)sh[a] : 0.0f; }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < APL; ++k) { int a = lane + 32 * k; if (a < A) shf[a] = mine[k]; }
        __syncwarp();
        float s = np_sum<float>(shf, A);
        probs_f64 = (s == 0.0f);  // np.zeros(len) is float64
#pragma unroll
        for (int k = 0; k < APL; ++k) probs[k] = (s != 0.0f) ? (double)__fdiv_rn(mine[k], s) : 0.0;
    }
    __syncwarp();
    bool out_f64;
#pragma unroll
    for (int k = 0; k < APL; ++k) {
        int a = lane + 32 * k;
        if (a >= A) continue;
        double r;
        if (probs_f64) {
            r = __dadd_rn(__dmul_rn(1.0 - coeff, probs[k]), __dmul_rn(coeff, noise ? noise[(int64_t)t * A + a] : 0.0));
        } else if (noise) {
            float c1 = (float)(1.0 - coeff);  // python float is "weak": float32 multiply
            r = __dadd_rn((double)__fmul_rn(c1, (float)probs[k]), __dmul_rn(coeff, noise[(int64_t)t * A + a]));
        } else {
            float c1 = (float)(1.0 - coeff), z = (float)__dmul_rn(coeff, 0.0);
            r = (double)__fadd_rn(__fmul_rn(c1, (float)probs[k]), z);
        }
        rp[a] = r;
    }
    out_f64 = probs_f64 || noise != nullptr;
    T.flags = (T.flags & ~(TF_PRIOR_F64 | TF_PREP_PENDING)) | TF_PRIOR_SET | (out_f64 ? TF_PRIOR_F64 : 0u);
    __syncwarp();
}

// One pending simulation as the backup needs it: the leaf's header copy, node index, path and net outputs.
// For lane 0 all of it is preloaded at kernel entry with loads whose addresses depend only on t (one round trip).
// Path element j (node j of the path root..leaf) lives on lane j & 31, slot j >> 5; a path is at most
// (number of real edges + 1) < 32 * APL nodes long.
template <int APL>
struct StepInputs {
    uint4 lh0, lh1;     // pending leaf header
    int leaf, plen;
    uint32_t pe[APL];   // parent << 8 | action | to_play << 31
    float w[APL];       // sequential mode: W and N of the node's own record (in its parent) before this simulation
    int n[APL];
    float p[APL];
    float value;
};

// Statistics of the simulations one launch finishes for a tree, flushed to the TreeRec once (sequential mode).
struct WaveStats {
    int sims, term, hits, path, maxdeep;
};

// `nrow` = row of the evaluator's batch (priors / values); the engine-owned pending record and path are indexed by
// slot and tree.  nrow < 0: k * n_trees + t (the non-compact layout).
template <int APL, bool SEQ>
__device__ __forceinline__ void load_pending(const Board& b, const TreeArgs& ta, int t, int k, int64_t nrow,
                                             const float* __restrict__ priors, const float* __restrict__ values,
                                             StepInputs<APL>& in, int lane) {
    const int64_t row = (int64_t)k * ta.n_trees + t;
    if (nrow < 0) nrow = row;
    const uint4* pr = ta.pend + row * 3;
    in.lh0 = pr[0]; in.lh1 = pr[1];
    const uint4 m = pr[2];
    in.leaf = (int)m.x; in.plen = (int)m.y;
#pragma unroll
    for (int i = 0; i < APL; ++i) {
        in.pe[i] = ta.path[row * PATH_CAP + lane + 32 * i];
        in.w[i] = 0.0f; in.n[i] = 0;
        if (SEQ) {
            const uint2 wn = ta.path_wn[(int64_t)t * PATH_CAP + lane + 32 * i];
            in.w[i] = __uint_as_float(wn.x); in.n[i] = (int)wn.y;
        }
    }
#pragma unroll
    for (int q = 0; q < APL; ++q) { int a = lane + 32 * q; in.p[q] = a < b.A ? priors[nrow * b.A + a] : 0.0f; }
    in.value = values[nrow];
}

// ---- evaluation cache (the engine's form of AsyncBatchedProxy's LRU, utils/proxies.py:23-26,35-43).
// Key = get_hash() = (edge set, boxes_to_close[to_play]) (dots_boxes_game.py:106-112): exactly what get_features()
// shows the net, so a hit returns what the net would return.  A 96-bit slice of the key sits in EVERY 16-byte cell next to
// its 4 payload bytes and a lookup only hits when all A cells carry their slice of the probe's key; cells are written with single
// 16-byte stores, so whatever races between trees of one launch (same key: same payload; different keys on one slot:
// mixed cells) can only turn a hit into a miss, never into a wrong evaluation.
// The key is 136 bits (128 edge bits for boards up to 7x7, 8 bits of 2 * boxes_to_close); a cell has room for 96, so even
// cells carry the slice {e0 lo, e0 hi, e1 lo} and odd cells {e1 hi, btc, table epoch}: a hit still needs EVERY cell to carry its slice
// of the probe's key, i.e. all 136 bits are compared (A / 2 times each).
// (k = the slice of THIS lane's cells, chosen by the lane's parity: a k[parity][3] array indexed at run time would live in
// local memory)
struct CacheKey { uint32_t k0, k1, k2; uint32_t slot; };
__device__ __forceinline__ CacheKey cache_key(const TreeArgs& ta, const Hdr& h, int par) {
    const int btc = h.to_play ? h.btc1 : h.btc0;
    CacheKey k;
    k.k0 = par ? (uint32_t)(h.e1 >> 32) : (uint32_t)h.e0;
    k.k1 = par ? ((uint32_t)btc & 0xffu) : (uint32_t)(h.e0 >> 32);
    k.k2 = par ? __ldg(ta.cache_epoch) : (uint32_t)h.e1;
    uint64_t x = h.e0 * 0x9E3779B97F4A7C15ull ^ (h.e1 + ((uint64_t)(btc & 0xff) << 56) + 0x632BE59BD9B4E019ull) * 0xC2B2AE3D27D4EB4Full;
    x ^= x >> 29; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 32;
    k.slot = (uint32_t)x & ta.cache_mask;
    return k;
}

// probe for the leaf in in.lh0/lh1; on a hit in.p / in.value hold the cached net outputs
template <int APL>
__device__ __forceinline__ bool cache_lookup(const Board& b, const TreeArgs& ta, StepInputs<APL>& in, int lane) {
    const Hdr h = unpack_hdr(in.lh0, in.lh1);
    const int par = lane & 1;  // a = lane + 32 k has the parity of the lane
    const CacheKey key = cache_key(ta, h, par);
    const uint4* cells = ta.cache + (size_t)key.slot * (size_t)b.A;
    uint4 c[APL];
    bool ok = true;
#pragma unroll
    for (int k = 0; k < APL; ++k) {
        const int a = lane + 32 * k;
        if (a < b.A) {
            c[k] = cells[a];
            ok = ok && c[k].y == key.k0 && c[k].z == key.k1 && c[k].w == key.k2;
        } else c[k] = make_uint4(0, 0, 0, 0);
    }
    if (!__all_sync(0xffffffffu, ok)) return false;
    const int vl = ta.cache_vcell & 31, vk = ta.cache_vcell >> 5;
    uint32_t vbits = 0;
#pragma unroll
    for (int k = 0; k < APL; ++k) {
        in.p[k] = __uint_as_float(c[k].x);
        if (k == vk) { vbits = c[k].x; if (lane == vl) in.p[k] = 0.0f; }  // a padding action: its prior is masked anyway
    }
    in.value = __uint_as_float(__shfl_sync(0xffffffffu, vbits, vl));
    return true;
}

template <int APL>
__device__ __forceinline__ void cache_insert(const Board& b, const TreeArgs& ta, const Hdr& lh, const StepInputs<APL>& in, int lane) {
    const int par = lane & 1;
    const CacheKey key = cache_key(ta, lh, par);
    uint4* cells = ta.cache + (size_t)key.slot * (size_t)b.A;
#pragma unroll
    for (int k = 0; k < APL; ++k) {
        const int a = lane + 32 * k;
        if (a < b.A) {
            const float payload = (a == ta.cache_vcell) ? in.value : in.p[k];
            cells[a] = make_uint4(__float_as_uint(payload), key.k0, key.k1, key.k2);
        }
    }
}

// expand + backup of one pending leaf (mcts.py:116-132 and the prior masking of 188-196).  The virtual loss was
// subtracted by the selection that produced the path (mcts.py:109), so every path node just gets
// W = fl32(W + fl32(v*s + 1)) and N += 1.
// NumPy's float32 add-reduce of a[0..A) (pairwise_sum, one block of < 128 elements: eight running sums over rows of
// eight, combined ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the tail) for a[lane + 32 k] = p[k], with shuffles:
// lane j < 8 accumulates r[j], three butterfly steps combine them in NumPy's order (float addition commutes), lane 0
// adds the tail; every lane returns the sum.  8 <= A <= 32 * APL.
template <int APL>
__device__ __forceinline__ float warp_np_sum(const float (&p)[APL], int A, int lane) {
    const int n8 = A & ~7;
    float r = 0.0f;
#pragma unroll
    for (int k = 0; k < APL; ++k)
#pragma unroll
        for (int mm = 0; mm < 4; ++mm) {
            const int base = 32 * k + 8 * mm;  // row of eight: elements base..base+7 live on lanes 8*mm..8*mm+7 of slot k
            if (base < n8) {
                const float v = __shfl_sync(0xffffffffu, p[k], (8 * mm + lane) & 31);
                r = (base == 0) ? v : __fadd_rn(r, v);
            }
        }
    r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 1));
    r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 2));
    r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 4));
#pragma unroll
    for (int q = 0; q < 7; ++q) {
        const int idx = n8 + q;
        if (idx < A) {
            float v = 0.0f;  // element idx sits on lane idx & 31 of slot idx >> 5; the slot is chosen AFTER the shuffles so that
                             // p[] is never indexed at run time
#pragma unroll
            for (int k = 0; k < APL; ++k) {
                const float vk = __shfl_sync(0xffffffffu, p[k], idx & 31);
                v = (k == (idx >> 5)) ? vk : v;
            }
            r = __fadd_rn(r, v);
        }
    }
    return __shfl_sync(0xffffffffu, r, 0);
}

// `src`: where in.p / in.value come from -- EV_NET (the evaluator: remembered in the eval cache if there is one),
// EV_CACHE (a cache hit), EV_NONE (terminal leaf, no evaluation).
enum { EV_NET = 0, EV_CACHE = 1, EV_NONE = 2 };
// SEQ (max_pending_evals == 1): nothing reads the tree between a selection and its backup, so the selection wrote no
// virtual loss and kept every path node's {W, N} in registers (in.w / in.n); the backup computes
// W = fl32(fl32(W - 1) + fl32(v*s + 1)) -- the reference's two roundings -- and N + 1 from those and stores them
// without re-reading the records; the leaf gets the +1 without the -1 (reference quirk).  Statistics go to `ws`.
// !SEQ: the records carry the virtual loss of all selections in flight; read-modify-write.
template <int APL, int NW, bool SEQ>
__device__ __forceinline__ void tree_expand_backup(const Board& b, const TreeArgs& ta, int t, TreeHot& T,
                                                   const StepInputs<APL>& in, double* sh, int lane, int src, WaveStats& ws) {
    const int A = b.A;
    char* lp = node_ptr(ta, t, in.leaf);
    Hdr lh = unpack_hdr(in.lh0, in.lh1);
    const bool terminal = lh.flags & NF_TERMINAL;
    float value;
    if (!terminal) {
        if (src == EV_NET && ta.cache) cache_insert<APL>(b, ta, lh, in, lane);
        // child_priors * valid (float32), NumPy-order sum, renormalise unless s == 1 or s <= 0
        float p[APL];
#pragma unroll
        for (int k = 0; k < APL; ++k) {
            int a = lane + 32 * k;
            p[k] = 0.0f;
            if (a < A) {
                const uint64_t ed = (NW == 1 || a < 64) ? lh.e0 : lh.e1;
                bool legal = ((b.real[NW == 1 ? 0 : (a >> 6)] & ~ed) >> (a & 63)) & 1ull;
                p[k] = legal ? in.p[k] : __fmul_rn(in.p[k], 0.0f);
            }
        }
        float s;
        if (SEQ) {
            s = warp_np_sum<APL>(p, A, lane);
        } else {
            float* shf = reinterpret_cast<float*>(sh);
#pragma unroll
            for (int k = 0; k < APL; ++k) { int a = lane + 32 * k; if (a < A) shf[a] = p[k]; }
            __syncwarp();
            s = np_sum<float>(shf, A);
            __syncwarp();
        }
        Child* ch = node_children(lp);
        const bool renorm = (s > 0.0f && s != 1.0f);
#pragma unroll
        for (int k = 0; k < APL; ++k) {
            int a = lane + 32 * k;
            if (a < A) {
                float q = renorm ? __fdiv_rn(p[k], s) : p[k];
                *reinterpret_cast<uint4*>(&ch[a]) = make_uint4(0u, 0u, __float_as_uint(q), 0u);  // {W=0, N=0, prior, child=none}
            }
        }
        value = in.value;
    } else {
        value = (float)lh.result;  // get_result(): python int 1 / 0
        if (in.leaf == 0) {
            // a terminal ROOT is re-expanded with np.zeros(A) on every visit (mcts.py:195-198), which
            // also discards whatever the UCT_search head mixed into its child_priors
            double* rp = ta.root_prior + (int64_t)t * A;
            for (int a = lane; a < A; a += 32) rp[a] = 0.0;
            T.flags |= TF_PRIOR_SET | TF_PRIOR_F64;
        }
    }
    if (!(lh.flags & NF_EXPANDED) && lane == 0) {
        lh.flags |= NF_EXPANDED;
        uint4 a4, b4;
        pack_hdr(lh, a4, b4);
        reinterpret_cast<uint4*>(lp)[1] = b4;
    }
    const int plen = in.plen;
#pragma unroll
    for (int i = 0; i < APL; ++i) {
        const int j = lane + 32 * i;
        if (j >= plen) continue;
        const uint32_t pe = in.pe[i];
        const int tp = pe >> 31;
        const float v = (tp == lh.to_play) ? value : -value;
        const float add = __fadd_rn(v, 1.0f);
        const bool had_vl = SEQ && j < plen - 1;  // every node the selection left behind (mcts.py:109)
        if (j == 0) {
            // only lane 0 reaches j == 0; T is written back by lane 0
            const float w0 = had_vl ? __fsub_rn(T.root_W, 1.0f) : T.root_W;
            T.root_W = __fadd_rn(w0, add);
            T.root_N += 1;
        } else {
            const int parent = (pe & 0x7fffffffu) >> 8, act = pe & 0xffu;
            float2* cell = reinterpret_cast<float2*>(&node_children(node_ptr(ta, t, parent))[act]);
            float2 wn;
            if (SEQ) {
                const float w0 = had_vl ? __fsub_rn(in.w[i], 1.0f) : in.w[i];
                wn.x = __fadd_rn(w0, add);
                wn.y = __int_as_float(in.n[i] + 1);
            } else {
                wn = *cell;
                wn.x = __fadd_rn(wn.x, add);
                wn.y = __int_as_float(__float_as_int(wn.y) + 1);
            }
            *cell = wn;
        }
    }
    if (SEQ) {
        ws.sims += 1;
        ws.term += terminal ? 1 : 0;
        ws.hits += (src == EV_CACHE) ? 1 : 0;
        ws.path += plen;
        ws.maxdeep = max(ws.maxdeep, lh.depth);
    } else if (lane == 0) {
        TreeRec* G = ta.trees + t;
        if (terminal) { G->terminal_count += 1; G->total_term += 1; }
        if (lh.depth > G->max_deepness) G->max_deepness = lh.depth;
        G->total_sims += 1;
        G->total_path += plen;
    }
}

// Warp argmax of (score, lowest action id wins ties) with three REDUX operations on an
// order-preserving integer image of the float64 score instead of 15 shuffles.
__device__ __forceinline__ int warp_argmax(double best, int best_a) {
    unsigned long long key = 0ull;
    if (best_a != 0x7fffffff) {
        unsigned long long u = (unsigned long long)__double_as_longlong(__dadd_rn(best, 0.0));  // -0.0 -> +0.0
        key = (u >> 63) ? ~u : (u | 0x8000000000000000ull);
    }
    const unsigned hi = (unsigned)(key >> 32), lo = (unsigned)key;
    const unsigned mh = __reduce_max_sync(0xffffffffu, hi);
    const bool c1 = (hi == mh) && best_a != 0x7fffffff;
    const unsigned ml = __reduce_max_sync(0xffffffffu, c1 ? lo : 0u);
    const bool c2 = c1 && lo == ml;
    return (int)__reduce_min_sync(0xffffffffu, c2 ? (unsigned)best_a : 0x7fffffffu);
}

// select_leaf with lazy child creation (mcts.py:105-114).  Returns the leaf kind (1 = needs evaluation,
// 2 = terminal, 0 = node pool exhausted); leaf header / index / path length are left in `out`.
// !SEQ (simulations in flight): VIRTUAL_LOSS is subtracted from every node left behind (mcts.py:109) -- the root's own
// W lives in the tree record (lane 0), any other node's in its parent's child record, which the lane that owned the
// winning action still holds from the previous level -- and the path goes to `path` (global) for the backup.
// SEQ (one simulation at a time): the loop stores nothing but a lazily created child; the path and each path node's
// {W, N} stay in registers (out.pe / out.w / out.n on lane == node index) and the backup applies the virtual loss.
template <int APL, int NW, bool SEQ>
__device__ __forceinline__ int tree_select(const Board& b, const TreeArgs& ta, int t, TreeHot& T,
                                           const LaneActions<APL, NW>& la, StepInputs<APL>& out, uint32_t* __restrict__ path,
                                           int lane) {
    const int A = b.A;
    const double* rp = ta.root_prior + (int64_t)t * A;
    int cur = 0, curN = T.root_N, depth = 0;
    int leaf = -1;
    Hdr leaf_hdr;
    char* const tree_base = node_ptr(ta, t, 0);
    float* vl_cell = nullptr;  // W of the current node's own record (valid on the lane that owned the action)
    float vl_w = 0.0f;
    while (true) {
        char* np = tree_base + (size_t)cur * (size_t)ta.stride;
        // header and child records are fetched together; an unexpanded / terminal node has garbage
        // child records, which are loaded but never interpreted
        const uint4* hp = reinterpret_cast<const uint4*>(np);
        const uint4 h0 = hp[0], h1 = hp[1];
        uint4 craw[APL];
#pragma unroll
        for (int k = 0; k < APL; ++k) {
            int a = lane + 32 * k;
            craw[k] = make_uint4(0, 0, 0, 0);
            if (a < A) craw[k] = hp[2 + a];
        }
        const double2 cs = puct_consts(ta, curN);
        double rprior[APL];
        if (depth == 0) {
#pragma unroll
            for (int k = 0; k < APL; ++k) { int a = lane + 32 * k; rprior[k] = a < A ? rp[a] : 0.0; }
        }
        const Hdr h = unpack_hdr(h0, h1);
        const bool interior = (h.flags & NF_EXPANDED) && !(h.flags & NF_TERMINAL);
        if (depth == 0 && lane == 0) {
            if (SEQ) out.pe[0] = PATH_ROOT | ((uint32_t)h.to_play << 31);
            else path[0] = PATH_ROOT | ((uint32_t)h.to_play << 31);
        }
        if (!interior) { leaf = cur; leaf_hdr = h; break; }
        if (!SEQ) {
            // current.total_value -= VIRTUAL_LOSS
            if (depth == 0) { if (lane == 0) T.root_W = __fsub_rn(T.root_W, 1.0f); }
            else if (vl_cell) *vl_cell = __fsub_rn(vl_w, 1.0f);
        }

        const Mask<NW> e = hdr_edges<NW>(h);
        const double c0 = cs.x, sq = cs.y;
        // ---- float32 pre-pass.  The float64 score of mcts.py:91-99 costs two divisions per lane on the critical path of
        // every level; almost always one child is ahead of the others by far more than float32 can blur.  sf approximates
        // the real value c0 sqrt(N) prior / (n + 1) +- W / (n + 1) with |sf - exact| <= 9 * 2^-24 (|ps| + |q|) (ps: float32
        // images of c0 and sqrt(N) and their product, the approximate reciprocal (two units), two products -- eight units of
        // relative size 2^-24; q: three; the sum: one; the float64 score itself is within 2^-50 of the real value),
        // ef = 2^-19 (|ps| + |q|) + 2^-100 leaves a factor of 3.5.  A child whose upper bound is below the
        // best lower bound can neither win nor tie.  If exactly ONE child remains it is the argmax; otherwise (ties,
        // near-ties, N = 0) the float64 scores of the remaining candidates decide, lowest action first, as before.
        const float c0sq = __fmul_rn((float)c0, (float)sq);
        float sf[APL], ef[APL];
        bool legal_k[APL];
        int ncl_k[APL];  // boxes each of this lane's actions would close (decides the child's sign and who moves next)
        float lo_max = -INFINITY;
#pragma unroll
        for (int k = 0; k < APL; ++k) {
            const int a = lane + 32 * k;
            legal_k[k] = la.real[k] && !mask_test(e, a < A ? a : 0);
            ncl_k[k] = 0; sf[k] = 0.0f; ef[k] = 0.0f;
            if (legal_k[k]) {
                ncl_k[k] = la.closes(k, e, a);
                float inv;  // MUFU.RCP: relative error <= 2^-23 (PTX rcp.approx.f32), two units of 2^-24 in the bound above
                asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"((float)((int)craw[k].y + 1)));
                const float pr = (depth == 0) ? (float)rprior[k] : __uint_as_float(craw[k].z);
                const float ps = __fmul_rn(__fmul_rn(c0sq, inv), pr);
                const float q = __fmul_rn(__uint_as_float(craw[k].x), inv);
                sf[k] = ncl_k[k] ? __fadd_rn(ps, q) : __fsub_rn(ps, q);
                ef[k] = __fmaf_rn(1.9073486328125e-6f, __fadd_rn(fabsf(ps), fabsf(q)), 7.888609052210118e-31f);
                lo_max = fmaxf(lo_max, __fsub_rn(sf[k], ef[k]));
            }
        }
        {
            const unsigned u = __float_as_uint(lo_max);
            const unsigned key = (u >> 31) ? ~u : (u | 0x80000000u);  // order-preserving image of the float
            const unsigned m = __reduce_max_sync(0xffffffffu, key);
            lo_max = __uint_as_float((m >> 31) ? (m & 0x7fffffffu) : ~m);
        }
        int n_cand = 0, a_single = 0;
        bool cand[APL];
#pragma unroll
        for (int k = 0; k < APL; ++k) {
            // a node without visits of its own (a re-used root restarts at N = 0, mcts.py:169-174) ranks by value alone and
            // its unvisited children tie at zero: no point in bounding, every legal child goes to the exact comparison
            cand[k] = legal_k[k] && (curN == 0 || __fadd_rn(sf[k], ef[k]) >= lo_max);
            const unsigned bal = __ballot_sync(0xffffffffu, cand[k]);
            if (bal) { n_cand += __popc(bal); a_single = (__ffs(bal) - 1) + 32 * k; }
        }
        int a;
        if (n_cand == 1) {
            a = a_single;
        } else {
            double best = -INFINITY;
            int best_a = 0x7fffffff;
#pragma unroll
            for (int k = 0; k < APL; ++k) {
                if (cand[k]) {
                    Child c;
                    c.W = __uint_as_float(craw[k].x); c.N = (int)craw[k].y; c.prior = __uint_as_float(craw[k].z);
                    const int sign = ncl_k[k] ? 1 : -1;
                    const double prior = (depth == 0) ? rprior[k] : (double)c.prior;
                    const double sc = ucb_score<APL, NW>(c0, sq, c, prior, sign);
                    if (best_a == 0x7fffffff || sc > best) { best = sc; best_a = lane + 32 * k; }
                }
            }
            a = warp_argmax(best, best_a);  // a non-terminal node always has a legal move
        }
        const int owner = a & 31, kk = a >> 5;
        int child = 0, childN = 0, ncl = 0;
        uint32_t childW = 0;
        vl_cell = nullptr;
#pragma unroll
        for (int k = 0; k < APL; ++k)
            if (k == kk) {
                child = (int)craw[k].w; childN = (int)craw[k].y; ncl = ncl_k[k]; childW = craw[k].x;
                if (!SEQ && lane == owner) { vl_cell = &node_children(np)[a].W; vl_w = __uint_as_float(craw[k].x); }
            }
        child = __shfl_sync(0xffffffffu, child, owner);
        childN = __shfl_sync(0xffffffffu, childN, owner);
        ncl = __shfl_sync(0xffffffffu, ncl, owner);
        const int child_tp = ncl ? h.to_play : 1 - h.to_play;
        ++depth;
        const uint32_t pe = ((uint32_t)cur << 8) | (uint32_t)a | ((uint32_t)child_tp << 31);
        if (SEQ) {
            childW = __shfl_sync(0xffffffffu, childW, owner);
#pragma unroll
            for (int i = 0; i < APL; ++i)
            {   // selects, not `if (i == ...) out.pe[i] = ...`: the compiler turns that into a run-time index and the path
                // registers into local memory
                const bool mine = i == (depth >> 5) && lane == (depth & 31);
                out.pe[i] = mine ? pe : out.pe[i];
                out.w[i] = mine ? __uint_as_float(childW) : out.w[i];
                out.n[i] = mine ? childN : out.n[i];
            }
        } else if (lane == 0) path[depth] = pe;
        if (child == 0) {
            // lazily create the child (mcts.py:53-54 -> BoxesState.play, dots_boxes_game.py:91-94)
            const int idx = T.n_nodes;
            if (idx >= ta.max_nodes) { T.flags |= TF_ERR_POOL; T.sims_left = 0; return 0; }
            T.n_nodes = idx + 1;
            Hdr ns = h;
            if (NW == 1 || a < 64) ns.e0 |= 1ull << (a & 63); else ns.e1 |= 1ull << (a & 63);
            ns.just_played = h.to_play;
            ns.to_play = child_tp;
            if (ncl) { if (h.to_play) ns.btc1 -= 2 * ncl; else ns.btc0 -= 2 * ncl; }
            const int r = hdr_result(ns);
            ns.flags = (r != DBAZ_RESULT_NONE) ? NF_TERMINAL : 0;
            ns.depth = h.depth + 1;
            ns.parent = cur; ns.parent_action = a; ns.result = r;
            if (lane == 0) store_hdr_regs(node_ptr(ta, t, idx), ns);
            if (lane == owner) node_children(np)[a].child = idx;
            leaf = idx; leaf_hdr = ns;
            break;
        }
        cur = child; curN = childN;
    }
    pack_hdr(leaf_hdr, out.lh0, out.lh1);
    out.leaf = leaf;
    out.plen = depth + 1;
    return (leaf_hdr.flags & NF_TERMINAL) ? 2 : 1;
}

// ---------------------------------------------------------------- kernels
constexpr int TREE_WARPS = 1;  // trees per CTA: one, so that a tree with a long chain holds up nobody's CTA slot

template <int APL, int NW>
__global__ void __launch_bounds__(TREE_WARPS * 32)
k_search_begin(Board b, TreeArgs ta, const int32_t* __restrict__ num_reads, const double* __restrict__ noise, double coeff) {
    __shared__ double sh_all[TREE_WARPS][DBAZ_MAX_ACTIONS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t = blockIdx.x * TREE_WARPS + warp;
    if (t >= ta.n_trees) return;
    const int nr = num_reads[t];
    if (nr == -3) return;  // this tree is in the middle of a search of its own: leave it alone
    TreeHot T = load_hot(ta.trees + t);
    T.n_pending = 0;
    T.flags &= ~TF_FIRST_WAVE;
    if (nr == -2) {
        // only the initial _search() of an unexpanded root (mcts.py:207-208), no prior mix: lets a host
        // caller draw its Dirichlet noise AFTER the root evaluation, in the reference's RNG order
        dbaz_state rh = load_hdr(node_ptr(ta, t, 0));
        T.sims_left = (rh.flags & NF_EXPANDED) ? 0 : 1;
        T.flags &= ~TF_PREP_PENDING;
    } else if (nr < 0) {
        T.sims_left = 0;
        T.flags &= ~TF_PREP_PENDING;
    } else {
        dbaz_state rh = load_hdr(node_ptr(ta, t, 0));
        if (rh.flags & NF_EXPANDED) {
            root_prior_mix<APL, NW>(b, ta, t, T, rh, noise, coeff, sh_all[warp], lane);
            T.sims_left = nr;
            T.flags |= TF_FIRST_WAVE;
        } else {
            T.flags |= TF_PREP_PENDING;  // mcts.py:207-208: one extra _search() first
            T.sims_left = nr + 1;
        }
    }
    if (lane == 0) {
        store_hot(ta.trees + t, T);
        if (T.sims_left > 0) atomicAdd(&ta.ctr[5], 1);  // busy trees at the start of the search (zeroed by the host)
    }
}

// Hand a selected leaf to the evaluator: planes / packed state into batch row `row`, the engine-side pending record
// (header copy, node index, path length; in sequential mode also the path registers) into slot `prow`.
template <int APL, int NW, bool SEQ>
__device__ __forceinline__ void emit_leaf(const Board& b, const TreeArgs& ta, const StepInputs<APL>& in, int64_t prow, int64_t row,
                                          void* __restrict__ planes, int dtype, int layout, dbaz_state* __restrict__ leaf_states,
                                          int lane) {
    const Hdr lh = unpack_hdr(in.lh0, in.lh1);
    write_planes_warp<NW>(b, hdr_edges<NW>(lh), (int)(int8_t)(lh.to_play ? lh.btc1 : lh.btc0), planes, row, dtype, layout, lane);
    if (SEQ) {
#pragma unroll
        for (int i = 0; i < APL; ++i) {  // entries beyond the path length are never read
            ta.path[prow * PATH_CAP + lane + 32 * i] = in.pe[i];
            ta.path_wn[prow * PATH_CAP + lane + 32 * i] = make_uint2(__float_as_uint(in.w[i]), (uint32_t)in.n[i]);
        }
    }
    if (lane == 0) {
        uint4* pr = ta.pend + prow * 3;
        pr[0] = in.lh0; pr[1] = in.lh1; pr[2] = make_uint4((uint32_t)in.leaf, (uint32_t)in.plen, 0u, 0u);
        if (leaf_states) {
            Hdr pub = lh;
            pub.flags = 0; pub.depth = 0; pub.parent = -1; pub.parent_action = -1;
            store_hdr_regs(reinterpret_cast<char*>(&leaf_states[row]), pub);
        }
    }
}

// max_pending_evals == 1: strictly sequential simulations.  The evaluation of the previous wave comes back, then the
// tree runs on for as long as its simulations need no evaluator: terminal leaves (mcts.py:194-196) and leaves found
// in the eval cache (the proxy returns those without suspending, utils/proxies.py:35-38) complete on the spot; the
// first leaf that needs the net ends the wave.  Returns true while the tree still has work.
template <int APL, int NW>
__device__ __forceinline__ bool search_step_seq(const Board& b, const TreeArgs& ta, int t,
                                                const float* __restrict__ priors, const float* __restrict__ values,
                                                const double* __restrict__ noise, double coeff, void* __restrict__ planes,
                                                int dtype, int layout, dbaz_state* __restrict__ leaf_states,
                                                int8_t* __restrict__ leaf_kind, double* sh, int lane) {
    // ---- one round trip: everything whose address depends only on t
    TreeHot T = load_hot(ta.trees + t);
    const bool compact = ta.compact;
    LaneActions<APL, NW> la;
    la.load(b, ta.act_tab, lane);
    StepInputs<APL> in;
    if (!compact) load_pending<APL, true>(b, ta, t, 0, -1, priors, values, in, lane);

    if (T.n_pending <= 0 && T.sims_left <= 0) {  // idle tree
        if (leaf_kind && !compact && lane == 0) leaf_kind[t] = 0;
        return false;
    }
    if (compact) load_pending<APL, true>(b, ta, t, 0, T.n_pending > 0 ? T.row : 0, priors, values, in, lane);
    WaveStats ws = {0, 0, 0, 0, 0};
    if (T.n_pending > 0) {
        tree_expand_backup<APL, NW, true>(b, ta, t, T, in, sh, lane, EV_NET, ws);
        T.n_pending = 0;
        T.root_N = __shfl_sync(0xffffffffu, T.root_N, 0);  // lane 0 owns the authoritative TreeRec
        __syncwarp();
        if (T.flags & TF_PREP_PENDING) {
            dbaz_state rh = load_hdr(node_ptr(ta, t, 0));
            root_prior_mix<APL, NW>(b, ta, t, T, rh, noise, coeff, sh, lane);
        }
    }
    T.flags &= ~TF_FIRST_WAVE;
    int inline_done = 0;
    // A launch lasts as long as its longest chain.  Bounding the chains by COUNT makes a tree whose simulations are cheap
    // (upper levels in L2, cache hits) stop as early as one whose every level waits for DRAM; bounding them by TIME lets
    // the cheap ones run on while the launch is waiting for the expensive ones anyway.  Results do not depend on where a
    // chain is cut (the next launch continues it), so the clock only shapes the schedule.
    const long long t_start = ta.chain_clk > 0 ? clock64() : 0ll;
    while (T.sims_left > 0) {
        __syncwarp();  // stores of the previous backup must be visible to this selection's loads
        const int kind = tree_select<APL, NW, true>(b, ta, t, T, la, in, nullptr, lane);
        if (!kind) break;  // node pool exhausted
        T.sims_left -= 1;
        int src = EV_NONE;
        if (kind == 1) {
            if (ta.cache && cache_lookup<APL>(b, ta, in, lane)) src = EV_CACHE;
            else {
                int64_t row = t;
                if (compact) {
                    int r = 0;
                    if (lane == 0) r = (int)(atomicAdd(reinterpret_cast<unsigned long long*>(ta.ctr), 1ull << 40) >> 40);
                    r = __shfl_sync(0xffffffffu, r, 0);
                    if (r >= ta.batch_rows) {
                        // the evaluator's batch is full: this selection is dropped and repeated in the next wave.
                        // It stored nothing but (possibly) the new child node, which the repeat walks into, so the
                        // repeat finds the same leaf over the same path.
                        T.sims_left += 1;
                        break;
                    }
                    T.row = r;
                    row = r;
                }
                emit_leaf<APL, NW, true>(b, ta, in, t, row, planes, dtype, layout, leaf_states, lane);
                T.n_pending = 1;
                break;
            }
        }
        tree_expand_backup<APL, NW, true>(b, ta, t, T, in, sh, lane, src, ws);
        T.root_N = __shfl_sync(0xffffffffu, T.root_N, 0);
        if (src == EV_CACHE && (T.flags & TF_PREP_PENDING)) {
            __syncwarp();
            dbaz_state rh = load_hdr(node_ptr(ta, t, 0));
            root_prior_mix<APL, NW>(b, ta, t, T, rh, noise, coeff, sh, lane);
        }
        if (ta.max_inline > 0 && ++inline_done >= ta.max_inline) break;
        if (ta.chain_clk > 0 && clock64() - t_start > (long long)ta.chain_clk) break;
    }
    if (lane == 0) {
        if (leaf_kind && !compact) leaf_kind[t] = (int8_t)T.n_pending;
        store_hot(ta.trees + t, T);
        if (ws.sims) {
            // tree statistics of the simulations this launch finished: reductions without a return value (RED), so the
            // warp does not wait for the old values of fields only this warp ever touches
            TreeRec* G = ta.trees + t;
            if (ws.term) { atomicAdd(&G->terminal_count, ws.term); atomicAdd(&G->total_term, ws.term); }
            atomicMax(&G->max_deepness, ws.maxdeep);
            atomicAdd(&G->total_sims, (uint32_t)ws.sims);
            if (ws.hits) atomicAdd(&G->cache_hits, (uint32_t)ws.hits);
            atomicAdd(&G->total_path, (unsigned long long)ws.path);
        }
    }
    return T.n_pending > 0 || T.sims_left > 0;
}

// max_pending_evals = K > 1: the reference's waves (mcts.py:228-242).  Returns true while the tree still has work.
template <int APL, int NW>
__device__ __forceinline__ bool search_step_waves(const Board& b, const TreeArgs& ta, int t, int pending,
                                                  const float* __restrict__ priors, const float* __restrict__ values,
                                                  const double* __restrict__ noise, double coeff, void* __restrict__ planes,
                                                  int dtype, int layout, dbaz_state* __restrict__ leaf_states,
                                                  int8_t* __restrict__ leaf_kind, double* sh, int lane) {
    // ---- one round trip: everything whose address depends only on t
    TreeHot T = load_hot(ta.trees + t);
    StepInputs<APL> in;
    load_pending<APL, false>(b, ta, t, 0, -1, priors, values, in, lane);
    LaneActions<APL, NW> la;
    la.load(b, ta.act_tab, lane);
    if (T.n_pending <= 0 && T.sims_left <= 0) {  // idle tree
        if (leaf_kind) for (int r = lane; r < pending; r += 32) leaf_kind[(int64_t)r * ta.n_trees + t] = 0;
        return false;
    }
    WaveStats ws = {0, 0, 0, 0, 0};  // unused: the statistics are updated in place
    // ---- the evaluations of the previous wave come back: expand + backup, in selection order
    const int n_back = T.n_pending;
    for (int k = 0; k < n_back; ++k) {
        if (k > 0) { __syncwarp(); load_pending<APL, false>(b, ta, t, k, -1, priors, values, in, lane); }
        tree_expand_backup<APL, NW, false>(b, ta, t, T, in, sh, lane, EV_NONE, ws);
    }
    T.n_pending = 0;
    if (n_back > 0) {
        // lane 0 owns the authoritative TreeRec; re-broadcast what the other lanes need
        T.root_N = __shfl_sync(0xffffffffu, T.root_N, 0);
        __syncwarp();
        if (T.flags & TF_PREP_PENDING) {
            dbaz_state rh = load_hdr(node_ptr(ta, t, 0));
            root_prior_mix<APL, NW>(b, ta, t, T, rh, noise, coeff, sh, lane);
            T.flags |= TF_FIRST_WAVE;
        }
    }
    // ---- this wave's selections.  Width: 1 while the root still awaits its own expansion (mcts.py:207-208), else
    // min(max_pending_evals, A) for the first wave of a search and max_pending_evals afterwards (mcts.py:228-236).
    int width = pending;
    if (T.flags & TF_PREP_PENDING) width = 1;
    else if (T.flags & TF_FIRST_WAVE) { width = min(pending, b.A); T.flags &= ~TF_FIRST_WAVE; }
    const int n_sel = min(width, T.sims_left);
    int n_out = 0;
    for (int k = 0; k < n_sel; ++k) {
        __syncwarp();  // stores of the backups / previous selections must be visible to this selection's loads
        const int64_t row = (int64_t)n_out * ta.n_trees + t;
        uint32_t* path = ta.path + row * PATH_CAP;
        const int kind = tree_select<APL, NW, false>(b, ta, t, T, la, in, path, lane);
        if (!kind) break;  // node pool exhausted
        T.sims_left -= 1;
        if (kind == 2) {
            // a terminal leaf never awaits the net: its simulation completes before the next one is selected
            __syncwarp();
#pragma unroll
            for (int i = 0; i < APL; ++i) in.pe[i] = path[lane + 32 * i];
            tree_expand_backup<APL, NW, false>(b, ta, t, T, in, sh, lane, EV_NONE, ws);
            T.root_N = __shfl_sync(0xffffffffu, T.root_N, 0);
            continue;
        }
        emit_leaf<APL, NW, false>(b, ta, in, row, row, planes, dtype, layout, leaf_states, lane);
        if (leaf_kind && lane == 0) leaf_kind[row] = 1;
        ++n_out;
    }
    T.n_pending = n_out;
    if (leaf_kind) for (int r = lane; r < pending; r += 32) if (r >= n_out) leaf_kind[(int64_t)r * ta.n_trees + t] = 0;
    if (lane == 0) store_hot(ta.trees + t, T);
    return T.n_pending > 0 || T.sims_left > 0;
}

// SEQ: max_pending_evals == 1 (search_step_seq); else the K-wave path.  Two kernels rather than one branch: each gets its
// own register allocation and half the code.
template <int APL, int NW, bool SEQ>
// Resident trees per SM (= register cap): 28 -> 72 registers for one action per lane (3x3), 20 -> 102 for two; for three and
// more (5x5: 168 registers uncapped, 12 trees per SM, 13 % of the warp slots) 16 -> 128 registers, even where that spills:
// the kernel is latency-bound with nine waves of CTAs, so residency wins -- 139 -> 114 us per launch on configs[3] (20 -> 96
// registers: 111 us, 156 bytes of spills).
__global__ void __launch_bounds__(TREE_WARPS * 32, (APL == 1 ? 28 : (APL == 2 ? 20 : 16)) / TREE_WARPS)
k_search_step(Board b, TreeArgs ta, int pending /* max_pending_evals of this search, <= ta.max_pending */,
              const float* __restrict__ priors, const float* __restrict__ values,
              const double* __restrict__ noise, double coeff, void* __restrict__ planes, int dtype, int layout,
              dbaz_state* __restrict__ leaf_states, int8_t* __restrict__ leaf_kind) {
    __shared__ double sh_all[TREE_WARPS][DBAZ_MAX_ACTIONS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t = blockIdx.x * TREE_WARPS + warp;
    bool busy = false;
    if (t < ta.n_trees) {
        if (SEQ)
            busy = search_step_seq<APL, NW>(b, ta, t, priors, values, noise, coeff, planes, dtype, layout, leaf_states, leaf_kind,
                                            sh_all[warp], lane);
        else
            busy = search_step_waves<APL, NW>(b, ta, t, pending, priors, values, noise, coeff, planes, dtype, layout, leaf_states,
                                              leaf_kind, sh_all[warp], lane);
    }
    // ---- wave bookkeeping, per warp (no CTA barrier: a warp leaves as soon as its tree is done, so a long chain keeps
    // one warp slot busy, not four).  Rows asked for, busy trees and finished warps share ONE 64-bit word, so a single
    // atomic per warp keeps them consistent without a fence; the warp that completes the count publishes and re-arms.
    if (lane == 0) {
        unsigned long long* word = reinterpret_cast<unsigned long long*>(ta.ctr);
        const unsigned long long inc = 1ull | (busy ? (1ull << 20) : 0ull);
        const unsigned long long now = atomicAdd(word, inc) + inc;
        if ((now & 0xfffffull) == (unsigned long long)(gridDim.x * TREE_WARPS)) {
            const int rows = (int)(now >> 40);
            ta.ctr[4] = rows;
            ta.ctr[5] = (int)((now >> 20) & 0xfffffull);
            if (rows > ta.ctr[6]) ta.ctr[6] = rows;
            *word = 0ull;  // nobody else touches it before the next launch
        }
    }
}

// UCT_search's time limit (mcts.py:232-233): launch no further simulations; pending leaves still back up
__global__ void k_search_stop(TreeArgs ta) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ta.n_trees) return;
    ta.trees[t].sims_left = 0;
    ta.trees[t].flags &= ~TF_PREP_PENDING;
}

// create_root_uct_node for every tree
__global__ void k_reset_roots(Board b, TreeArgs ta, const dbaz_state* __restrict__ roots) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ta.n_trees) return;
    dbaz_state s;
    if (roots) s = roots[t];
    else state_init(b, s);  // empty board
    int r = state_result(s);
    s.flags = (r != DBAZ_RESULT_NONE) ? NF_TERMINAL : 0;
    s.depth = 1;  // TreeRoot.deepness (0) + 1, mcts.py:64-65
    s.parent = -1; s.parent_action = -1; s.result = (int16_t)r;
    store_hdr(node_ptr(ta, t, 0), s);
    TreeRec T;
    T.n_nodes = 1; T.root_N = 0; T.root_W = 0.0f; T.sims_left = 0; T.n_pending = 0; T.row = 0; T.flags = 0;
    T.max_deepness = 0; T.deepness_correction = 0; T.terminal_count = 0; T.tree_size = 0; T.total_term = 0;
    T.total_sims = 0; T.cache_hits = 0; T.total_path = 0;
    ta.trees[t] = T;
}

// init_mcts_tree (mcts.py:163-180).  One CTA per tree.  With reuse the kept subtree is compacted
// in place: (1) reachability by parent pointers (a child always has a larger index than its
// parent, so a fixed point over "marked[parent]" converges in <= height rounds, in shared
// memory); (2) prefix sum of the mark bits gives new indices; (3) nodes move front-to-back in
// chunks of one node per warp (all loads of a chunk complete before its stores; new <= old so
// nothing unread is overwritten), remapping parent and child indices on the fly.
constexpr int ADV_THREADS = 1024;  // the most threads a launch may use; the launch picks 256 or 1024 (blockDim.x)
template <int NW>
__global__ void __launch_bounds__(ADV_THREADS)
k_advance_roots(Board b, TreeArgs ta, const int32_t* __restrict__ moves, int reuse) {
    extern __shared__ uint32_t smem_u32[];
    const int t = blockIdx.x;
    const int mv = moves[t];
    if (mv < 0) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthreads = blockDim.x;
    const int nwords = (ta.max_nodes + 31) >> 5;
    uint32_t* mark = smem_u32;                 // [nwords]
    uint32_t* prefix = smem_u32 + nwords;      // [nwords]
    uint16_t* parent16 = reinterpret_cast<uint16_t*>(smem_u32 + 2 * nwords);  // [max_nodes]
    __shared__ int s_changed, s_total;
    __shared__ TreeRec sT;
    __shared__ dbaz_state s_root;
    __shared__ Child s_entry;

    if (tid == 0) {
        sT = ta.trees[t];
        s_root = load_hdr(node_ptr(ta, t, 0));
        if (mv < b.A) s_entry = node_children(node_ptr(ta, t, 0))[mv];
    }
    __syncthreads();
    TreeRec T = sT;
    dbaz_state rh = s_root;
    if (!state_legal<NW>(b, rh, mv)) {
        if (tid == 0) { T.flags |= TF_ERR_MOVE; ta.trees[t] = T; }
        return;
    }
    const bool root_interior = (rh.flags & NF_EXPANDED) && !(rh.flags & NF_TERMINAL);
    const int child = root_interior ? s_entry.child : 0;
    const int nb_visits = root_interior ? s_entry.N : 0;
    const int n = T.n_nodes;
    if (tid == 0) atomicMax(&ta.ctr[7], n);  // high-water mark of the node pools (dbaz_search_status)

    if (child == 0 || !reuse) {
        if (tid == 0) {
            Mask<NW> box[2]; int lc[2][2];
            action_boxes<NW>(b, mv, box, lc);
            Mask<NW> e = load_edges<NW>(rh);
            mask_set(e, mv);
            dbaz_state ns = rh;
            state_apply<NW>(ns, mv, closed_count<NW>(e, box));
            int r = state_result(ns);
            ns.flags = (r != DBAZ_RESULT_NONE) ? NF_TERMINAL : 0;
            ns.depth = reuse ? rh.depth + 1 : 1;
            ns.parent = -1; ns.parent_action = (int16_t)mv; ns.result = (int16_t)r;
            store_hdr(node_ptr(ta, t, 0), ns);
            T.n_nodes = 1;
            T.deepness_correction = reuse ? ns.depth : 0;
            T.tree_size = reuse ? nb_visits : 0;
        }
    } else {
        for (int w = tid; w < nwords; w += nthreads) mark[w] = 0;
        for (int i = tid; i < n; i += nthreads) {
            int p = reinterpret_cast<const dbaz_state*>(node_ptr(ta, t, i))->parent;
            parent16[i] = (uint16_t)(p < 0 ? 0 : p);
        }
        __syncthreads();
        if (tid == 0) mark[child >> 5] = 1u << (child & 31);
        __syncthreads();
        while (true) {
            if (tid == 0) s_changed = 0;
            __syncthreads();
            for (int i = child + 1 + tid; i < n; i += nthreads) {
                if (!((mark[i >> 5] >> (i & 31)) & 1u)) {
                    int p = parent16[i];
                    if ((mark[p >> 5] >> (p & 31)) & 1u) { atomicOr(&mark[i >> 5], 1u << (i & 31)); s_changed = 1; }
                }
            }
            __syncthreads();
            if (!s_changed) break;
            __syncthreads();
        }
        if (tid == 0) {  // nwords <= 1024: a serial scan is a few microseconds
            int acc = 0;
            for (int w = 0; w < nwords; ++w) { prefix[w] = acc; acc += __popc(mark[w]); }
            s_total = acc;
        }
        __syncthreads();
        auto newidx = [&](int i) { return (int)(prefix[i >> 5] + __popc(mark[i >> 5] & ((1u << (i & 31)) - 1u))); };
        const int pieces = ta.stride >> 4;  // 16-byte pieces per node: 2 header + A children
        const int NWARPS = nthreads >> 5;
        constexpr int MAXP = (2 + DBAZ_MAX_ACTIONS + 31) / 32;
        for (int base = child; base < n; base += NWARPS) {
            const int i = base + warp;
            const bool live = i < n && ((mark[i >> 5] >> (i & 31)) & 1u);
            int4 buf[MAXP];
            int npc = 0;
            if (live) {
                const int4* src = reinterpret_cast<const int4*>(node_ptr(ta, t, i));
                const uint8_t fl = reinterpret_cast<const dbaz_state*>(src)->flags;
                // unexpanded / terminal nodes have no meaningful child records: move the header only
                npc = ((fl & NF_EXPANDED) && !(fl & NF_TERMINAL)) ? pieces : 2;
#pragma unroll
                for (int q = 0; q < MAXP; ++q) {
                    int pc = lane + 32 * q;
                    if (pc < npc) {
                        int4 v = src[pc];
                        if (pc == 1) v.z = (i == child) ? -1 : newidx(v.z);   // header.parent
                        else if (pc >= 2 && v.w != 0) v.w = newidx(v.w);      // Child.child
                        buf[q] = v;
                    }
                }
            }
            __syncthreads();
            if (live) {
                int4* dst = reinterpret_cast<int4*>(node_ptr(ta, t, newidx(i)));
#pragma unroll
                for (int q = 0; q < MAXP; ++q) {
                    int pc = lane + 32 * q;
                    if (pc < npc) dst[pc] = buf[q];
                }
            }
            __syncthreads();
        }
        if (tid == 0) {
            T.n_nodes = s_total;
            T.deepness_correction = reinterpret_cast<const dbaz_state*>(node_ptr(ta, t, 0))->depth;
            T.tree_size = nb_visits;
        }
    }
    if (tid == 0) {
        T.root_N = 0; T.root_W = 0.0f; T.n_pending = 0; T.sims_left = 0;
        T.max_deepness = 0; T.terminal_count = 0;
        T.flags &= ~(TF_PRIOR_SET | TF_PRIOR_F64 | TF_PREP_PENDING | TF_FIRST_WAVE);
        ta.trees[t] = T;
    }
}

// ------------------------------------------------------------ root views
// root.child_number_visits (mcts.py:244): one warp per tree, coalesced row store
__global__ void k_root_visits(Board b, TreeArgs ta, int32_t* __restrict__ out) {
    int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= ta.n_trees) return;
    char* np = node_ptr(ta, w, 0);
    dbaz_state h = load_hdr(np);
    bool interior = (h.flags & NF_EXPANDED) && !(h.flags & NF_TERMINAL);
    const Child* ch = node_children(np);
    for (int a = lane; a < b.A; a += 32) out[(int64_t)w * b.A + a] = interior ? ch[a].N : 0;
}

template <int NW>
__global__ void k_root_children(Board b, TreeArgs ta, float* __restrict__ W, double* __restrict__ priors,
                                int32_t* __restrict__ sign, double* __restrict__ ucb) {
    int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= ta.n_trees) return;
    const int A = b.A;
    char* np = node_ptr(ta, w, 0);
    dbaz_state h = load_hdr(np);
    TreeRec T = ta.trees[w];
    bool interior = (h.flags & NF_EXPANDED) && !(h.flags & NF_TERMINAL);
    const Child* ch = node_children(np);
    Mask<NW> e = load_edges<NW>(h);
    const double2 cs = puct_consts(ta, T.root_N);
    double c0 = cs.x, sq = cs.y;
    for (int a = lane; a < A; a += 32) {
        Child c; c.W = 0.0f; c.N = 0; c.prior = 0.0f; c.child = 0;
        if (interior) c = ch[a];
        double pr = (T.flags & TF_PRIOR_SET) ? ta.root_prior[(int64_t)w * A + a] : (double)c.prior;
        int sg = 1;  // child_player_changed defaults to +1 until the child is expanded (mcts.py:61-62,119)
        if (c.child != 0) {
            dbaz_state chd = load_hdr(node_ptr(ta, w, c.child));
            if (chd.flags & NF_EXPANDED) sg = (chd.to_play == (uint8_t)chd.just_played) ? 1 : -1;
        }
        int64_t o = (int64_t)w * A + a;
        if (W) W[o] = c.W;
        if (priors) priors[o] = pr;
        if (sign) sign[o] = sg;
        if (ucb) ucb[o] = ucb_score<1, NW>(c0, sq, c, pr, sg);
    }
    (void)e;
}

// Any node of one tree for walks from the host (UCTNode.children / print_mcts_tree, mcts.py:47-65,247-272): the node's
// state, its per-child arrays, the UCB scores children_ucb_score() would return for it, and its own N / W (which live in
// its parent's child record, or in the tree record for node 0).  One warp.
template <int NW>
__global__ void k_node_view(Board b, TreeArgs ta, int tree, int node, dbaz_state* __restrict__ state_out, float* __restrict__ W,
                            int32_t* __restrict__ N, double* __restrict__ priors, int32_t* __restrict__ child, int32_t* __restrict__ sign,
                            double* __restrict__ ucb, int32_t* __restrict__ own8, float* __restrict__ own_W) {
    const int lane = threadIdx.x & 31;
    const int A = b.A;
    TreeRec T = ta.trees[tree];
    if (node < 0 || node >= T.n_nodes) {
        if (lane == 0) own8[7] = 1;  // no such node
        return;
    }
    char* np = node_ptr(ta, tree, node);
    dbaz_state h = load_hdr(np);
    const bool interior = (h.flags & NF_EXPANDED) && !(h.flags & NF_TERMINAL);
    const Child* ch = node_children(np);
    int ownN = T.root_N;
    float ownW = T.root_W;
    if (node != 0) {
        const Child pc = node_children(node_ptr(ta, tree, h.parent))[h.parent_action];
        ownN = pc.N; ownW = pc.W;
    }
    const double2 cs = puct_consts(ta, ownN);
    for (int a = lane; a < A; a += 32) {
        Child c; c.W = 0.0f; c.N = 0; c.prior = 0.0f; c.child = 0;
        if (interior) c = ch[a];
        const double pr = (node == 0 && (T.flags & TF_PRIOR_SET)) ? ta.root_prior[(int64_t)tree * A + a] : (double)c.prior;
        int sg = 1;  // child_player_changed defaults to +1 until the child is expanded (mcts.py:61-62,119)
        if (c.child != 0) {
            dbaz_state chd = load_hdr(node_ptr(ta, tree, c.child));
            if (chd.flags & NF_EXPANDED) sg = (chd.to_play == (uint8_t)chd.just_played) ? 1 : -1;
        }
        W[a] = c.W; N[a] = c.N; priors[a] = pr; child[a] = c.child; sign[a] = sg;
        ucb[a] = ucb_score<1, NW>(cs.x, cs.y, c, pr, sg);
    }
    if (lane == 0) {
        own8[0] = ownN; own8[1] = (h.flags & NF_EXPANDED) ? 1 : 0; own8[2] = (h.flags & NF_TERMINAL) ? 1 : 0;
        own8[3] = h.parent; own8[4] = h.parent_action; own8[5] = h.depth; own8[6] = T.n_nodes; own8[7] = 0;
        *own_W = ownW;
        dbaz_state pub = h;
        pub.flags = 0; pub.depth = 0; pub.parent = -1; pub.parent_action = -1; pub.result = (int16_t)state_result(h);
        *state_out = pub;
    }
}

__global__ void k_tree_stats(TreeArgs ta, int32_t* __restrict__ stats8, float* __restrict__ root_W, float* __restrict__ q) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ta.n_trees) return;
    TreeRec T = ta.trees[t];
    dbaz_state h = load_hdr(node_ptr(ta, t, 0));
    if (stats8) {
        int32_t* o = stats8 + (int64_t)t * 8;
        o[0] = T.root_N; o[1] = T.max_deepness - T.deepness_correction; o[2] = T.tree_size; o[3] = T.terminal_count;
        o[4] = (h.flags & NF_EXPANDED) ? 1 : 0; o[5] = (h.flags & NF_TERMINAL) ? 1 : 0; o[6] = T.n_nodes;
        o[7] = (int32_t)(T.flags & (TF_ERR_POOL | TF_ERR_MOVE));
    }
    if (root_W) root_W[t] = T.root_W;
    if (q) q[t] = __fdiv_rn(T.root_W, (float)(1 + T.root_N));  // mcts.py:35
}

// 1 while a tree has simulations left or a leaf waiting for the evaluator
__global__ void k_tree_busy(TreeArgs ta, int8_t* __restrict__ out) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ta.n_trees) return;
    const TreeHot T = load_hot(ta.trees + t);
    out[t] = (T.sims_left > 0 || T.n_pending > 0) ? 1 : 0;
}

__global__ void k_root_states(TreeArgs ta, dbaz_state* __restrict__ out) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ta.n_trees) return;
    dbaz_state h = load_hdr(node_ptr(ta, t, 0));
    h.flags = 0; h.depth = 0; h.parent = -1; h.parent_action = -1; h.result = (int16_t)state_result(h);
    out[t] = h;
}

// dbaz_cache_clear: a new epoch (never 0xffffffff, the fill value of an empty cell)
__global__ void k_cache_epoch(uint32_t* epoch, uint32_t value) { *epoch = value; }

// {errored trees, total sims, total path nodes, max n_nodes, terminal leaves} by atomics (zeroed by the host)
__global__ void k_status(TreeArgs ta, unsigned long long* __restrict__ out4) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ta.n_trees) return;
    TreeRec T = ta.trees[t];
    if (T.flags & (TF_ERR_POOL | TF_ERR_MOVE)) atomicAdd(&out4[0], 1ull);
    atomicAdd(&out4[1], (unsigned long long)T.total_sims);
    atomicAdd(&out4[5], (unsigned long long)T.cache_hits);
    atomicAdd(&out4[2], T.total_path);
    atomicMax(&out4[3], (unsigned long long)max(T.n_nodes, t == 0 ? ta.ctr[7] : 0));
    atomicAdd(&out4[4], (unsigned long long)T.total_term);
}

}  // namespace dbaz
