// dbaz_capi.cu -- the extern "C" boundary declared in include/dbaz_b200.h.
// Plain pointers and sizes only; no torch types.  Built in-tree for sm_100a:
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC ...
#include <algorithm>
#include <numeric>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "dbaz_game_kernels.cuh"
#include "dbaz_nn_kernels.cuh"
#include "dbaz_tree_kernels.cuh"
#include "dbaz_selfplay.cuh"
#include "dbaz_tower.cuh"
#include "dbaz_loop.cuh"

using namespace dbaz;

struct dbaz_engine {
    dbaz_config cfg;
    Board board;
    TreeArgs ta;
    int apl, nw;
    int n_sms;
    size_t adv_smem;
    int adv_threads;   // threads per tree of k_advance_roots
    const double* noise;  // caller-owned device buffer of the current search (may be null)
    double coeff;
    int pending;          // max_pending_evals of the current search
    int cache_log2;       // log2(entries) of the eval cache, 0 = none
    uint32_t* d_cache_epoch;   // the table epoch the step kernels read (TreeArgs::cache_epoch)
    uint32_t cache_epoch;      // its value after the last dbaz_cache_clear / dbaz_cache_configure
    unsigned long long* d_status;
    int* d_tower_err;     // set by k_resnet_tower when a barrier wait times out
    long long* tower_dbg; // caller-owned timeline buffer (dbaz_nn_tower_trace), may be null
    std::string err;
};

static std::string g_create_err;

namespace {

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int fail(dbaz_engine* e, const std::string& msg) {
    if (e) e->err = msg; else g_create_err = msg;
    return 1;
}
int cuda_fail(dbaz_engine* e, const char* what, cudaError_t st) {
    return fail(e, std::string(what) + ": " + cudaGetErrorString(st));
}

#define DBAZ_CK(e, call)                                   \
    do {                                                   \
        cudaError_t st_ = (call);                          \
        if (st_ != cudaSuccess) return cuda_fail((e), #call, st_); \
    } while (0)

inline cudaStream_t S(uint64_t h) { return reinterpret_cast<cudaStream_t>(h); }
inline int blocks_for(int64_t n, int per) { return (int)((n + per - 1) / per); }

int upload_lut(dbaz_engine* e) {
    // c0(N) = log((N + base + 1) / base) + cpuct with the host libm -- the same function CPython's
    // math.log calls (mcts.py:92-93) -- so no device log ulp difference can flip an argmax.
    // sqrt(N) rides along in the same 16-byte entry (IEEE sqrt is correctly rounded on both sides).
    std::vector<double2> lut(e->ta.lut_size);
    for (int n = 0; n < e->ta.lut_size; ++n) {
        lut[n].x = std::log(((double)n + e->ta.cpuct_base + 1.0) / e->ta.cpuct_base) + e->ta.cpuct;
        lut[n].y = std::sqrt((double)n);
    }
    DBAZ_CK(e, cudaMemcpy(const_cast<double2*>(e->ta.lut), lut.data(), lut.size() * sizeof(double2), cudaMemcpyHostToDevice));
    return 0;
}

int launch_ok(dbaz_engine* e, const char* what) {
    cudaError_t st = cudaGetLastError();
    if (st != cudaSuccess) return cuda_fail(e, what, st);
    return 0;
}

}  // namespace

// dispatch on (actions per lane, mask words)
#define DBAZ_DISPATCH(e, EXPR)                                   \
    do {                                                         \
        if ((e)->apl == 1) { constexpr int APL = 1, NW = 1; EXPR; } \
        else if ((e)->apl == 2) { constexpr int APL = 2, NW = 1; EXPR; } \
        else if ((e)->apl == 3) { constexpr int APL = 3, NW = 2; EXPR; } \
        else { constexpr int APL = 4, NW = 2; EXPR; }            \
    } while (0)

template <typename T>
static int launch_stem(dbaz_engine* e, const dbaz_state* leaves, const float* w01, const float* Bp, const float* K2,
                       const float* scale, const float* shift, T* out, int n, int cout, int mode, cudaStream_t st) {
    const int H = e->board.rows, W = e->board.cols;
    const int groups = cout / 8, per_block = 128 / groups;
    const size_t smem = (size_t)((18 + 2 * H * W) * cout + 2 * cout) * sizeof(float);
    const int resident = std::max(1, (int)std::min<size_t>(4, (200 * 1024) / smem));
    const int grid = std::max(1, std::min((n + per_block - 1) / per_block, e->n_sms * resident));
#define DBAZ_STEM(HH, WW)                                                                                               \
    if (H == HH && W == WW) {                                                                                           \
        cudaFuncSetAttribute(k_nn_stem<T, HH, WW, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
        cudaFuncSetAttribute(k_nn_stem<T, HH, WW, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
        if (mode == 0) k_nn_stem<T, HH, WW, 0><<<grid, 128, smem, st>>>(leaves, w01, Bp, K2, scale, shift, out, n, cout); \
        else k_nn_stem<T, HH, WW, 1><<<grid, 128, smem, st>>>(leaves, w01, Bp, K2, scale, shift, out, n, cout);          \
        return launch_ok(e, "k_nn_stem");                                                                               \
    }
    DBAZ_STEM(4, 4)
    DBAZ_STEM(6, 6)
    DBAZ_STEM(3, 3)
    DBAZ_STEM(5, 5)
#undef DBAZ_STEM
    return fail(e, "dbaz_nn_stem: no specialisation for this board size (3x3, 5x5, 2x2, 4x4 boxes are built)");
}

template <typename T, int NT>
static int launch_stem_mma_nt(dbaz_engine* e, const dbaz_state* leaves, const T* w48, T* out, int64_t n, int cout, cudaStream_t st, StemPlanar pl) {
    const int H = e->board.rows, W = e->board.cols, HW = H * W;
    const size_t smem = (size_t)(cout / 8) * 3 * 32 * sizeof(uint2) + (size_t)((HW * STEM_K + 15) & ~15) +
                        (size_t)STEM_WARPS * 16 * (8 * (NT >= 16 ? NT / 2 : NT) * 2 + 16);
    const int64_t items = ((n * HW + 15) / 16) * (cout / (8 * NT));
    const int resident = (int)std::max<size_t>(1, std::min<size_t>(5, (200 * 1024) / smem));
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((items + STEM_WARPS - 1) / STEM_WARPS, (int64_t)e->n_sms * resident));
    cudaError_t rc = cudaFuncSetAttribute(k_nn_stem_mma<T, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(k_nn_stem_mma)", rc);
    k_nn_stem_mma<T, NT><<<grid, STEM_WARPS * 32, smem, st>>>(leaves, w48, out, (int)n, cout, H, W, pl);
    return launch_ok(e, "k_nn_stem_mma");
}

template <typename T>
static int launch_stem_mma(dbaz_engine* e, const dbaz_state* leaves, const T* w48, T* out, int64_t n, int cout, cudaStream_t st,
                           StemPlanar pl = StemPlanar{0, 0, 0, 0}) {
    // one work item = 16 rows x (8 * NT) channels; all channels in one item when cout <= 256 (A fragments built once)
    if (cout % 256 == 0) return launch_stem_mma_nt<T, 32>(e, leaves, w48, out, n, cout, st, pl);
    if (cout % 128 == 0) return launch_stem_mma_nt<T, 16>(e, leaves, w48, out, n, cout, st, pl);
    return launch_stem_mma_nt<T, 8>(e, leaves, w48, out, n, cout, st, pl);
}

extern "C" {

int dbaz_abi_version(void) { return DBAZ_ABI_VERSION; }
int dbaz_sizeof_state(void) { return (int)sizeof(dbaz_state); }

const char* dbaz_last_error(const dbaz_engine* e) { return e ? e->err.c_str() : g_create_err.c_str(); }

int dbaz_engine_create(const dbaz_config* cfg, dbaz_engine** out) {
    if (!cfg || !out) return fail(nullptr, "null argument");
    *out = nullptr;
    if (cfg->abi_version != DBAZ_ABI_VERSION) return fail(nullptr, "ABI version mismatch");
    const int L = cfg->board_l, C = cfg->board_c;
    if (L < 1 || C < 1) return fail(nullptr, "board dimensions must be >= 1");
    const int A = 2 * (L + 1) * (C + 1);
    if (A > DBAZ_MAX_ACTIONS) return fail(nullptr, "board too large: 2*(L+1)*(C+1) must be <= 128");
    if (L * C > 16000) return fail(nullptr, "board too large");
    if (cfg->n_games < 1 || cfg->n_games >= (1 << 20)) return fail(nullptr, "n_games must be in [1, 2^20) (trees per engine; game-rule calls take any n)");
    if (cfg->max_nodes < 2 || cfg->max_nodes > 65536) return fail(nullptr, "max_nodes must be in [2, 65536]");
    const int max_pending = cfg->max_pending > 0 ? cfg->max_pending : 1;
    if (max_pending > DBAZ_MAX_PENDING) return fail(nullptr, "max_pending too large");
    int ndev = 0;
    cudaError_t st = cudaGetDeviceCount(&ndev);
    if (st != cudaSuccess || ndev == 0)
        return fail(nullptr, std::string("no CUDA device: this engine has no CPU fallback (") + cudaGetErrorString(st) + ")");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, "bad device ordinal");
    DeviceGuard guard(cfg->device);

    dbaz_engine* e = new dbaz_engine();
    e->cfg = *cfg;
    Board& b = e->board;
    b.L = L; b.C = C; b.rows = L + 1; b.cols = C + 1; b.plane = b.rows * b.cols; b.A = A; b.nboxes = L * C; b.F = 3 * b.plane;
    b.real[0] = b.real[1] = 0;
    for (int a = 0; a < A; ++a) {
        int p = a / b.plane, rem = a % b.plane, l = rem / b.cols, c = rem % b.cols;
        bool real = p == 0 ? (c < C) : (l < L);
        if (real) b.real[a >> 6] |= 1ull << (a & 63);
    }
    e->apl = (A + 31) / 32;
    e->nw = A > 64 ? 2 : 1;
    cudaDeviceProp prop;
    if ((st = cudaGetDeviceProperties(&prop, cfg->device)) != cudaSuccess) { cuda_fail(nullptr, "cudaGetDeviceProperties", st); delete e; return 1; }
    e->n_sms = prop.multiProcessorCount;

    TreeArgs& ta = e->ta;
    std::memset(&ta, 0, sizeof(ta));
    ta.n_trees = cfg->n_games;
    ta.max_nodes = cfg->max_nodes;
    ta.stride = 32 + 16 * A;
    ta.max_pending = max_pending;
    e->pending = 1;
    // A node's visit count is bounded by the simulations that can pass through it: with tree reuse at most (moves of a game) x
    // (simulations per search), and a search cannot run more simulations than the node pool holds.  The default table covers
    // 128 x (pool size) visits (a 7x7 board has 112 moves), so the device-log fallback of puct_consts() is out of reach.
    ta.lut_size = cfg->lut_size > 0 ? cfg->lut_size
                                    : (int)std::max<int64_t>(65536, std::min<int64_t>((int64_t)1 << 23, 128 * ((int64_t)cfg->max_nodes + 1)));
    ta.cpuct = cfg->cpuct;
    ta.cpuct_base = cfg->cpuct_base;
    const size_t arena_bytes = (size_t)ta.n_trees * ta.max_nodes * ta.stride;
    auto alloc = [&](void** p, size_t bytes, const char* what) -> bool {
        cudaError_t s2 = cudaMalloc(p, bytes);
        if (s2 != cudaSuccess) {
            char buf[256];
            std::snprintf(buf, sizeof buf, "cudaMalloc(%s, %zu bytes): %s", what, bytes, cudaGetErrorString(s2));
            g_create_err = buf;
            return false;
        }
        return true;
    };
    bool ok = alloc((void**)&ta.arena, arena_bytes, "node pool") &&
              alloc((void**)&ta.trees, (size_t)ta.n_trees * sizeof(TreeRec), "tree table") &&
              alloc((void**)&ta.root_prior, (size_t)ta.n_trees * A * sizeof(double), "root priors") &&
              alloc((void**)&ta.path, (size_t)max_pending * ta.n_trees * PATH_CAP * sizeof(uint32_t), "paths") &&
              alloc((void**)&ta.path_wn, (size_t)ta.n_trees * PATH_CAP * sizeof(uint2), "path statistics") &&
              alloc((void**)&ta.lut, (size_t)ta.lut_size * sizeof(double2), "log/sqrt table") &&
              alloc((void**)&ta.act_tab, (size_t)A * 2 * sizeof(uint4), "action table") &&
              alloc((void**)&ta.pend, (size_t)max_pending * ta.n_trees * 3 * sizeof(uint4), "pending leaves") &&
              alloc((void**)&ta.ctr, 16 * sizeof(int), "wave counters") &&
              alloc((void**)&e->d_status, 8 * sizeof(unsigned long long), "status");
    if (!ok) { dbaz_engine_destroy(e); return 1; }
    if (upload_lut(e)) { g_create_err = e->err; dbaz_engine_destroy(e); return 1; }

    const int nwords = (ta.max_nodes + 31) >> 5;
    e->adv_smem = (size_t)2 * nwords * 4 + (size_t)ta.max_nodes * 2;
    // re-rooting one tree is a chain of block-wide phases: 1024 threads make it short (what the asynchronous loop of a few
    // thousand games waits for at every check); with tens of thousands of trees the launch is bound by how many trees are
    // resident at once, and 256 threads per tree put four times as many on an SM
    e->adv_threads = ta.n_trees >= 16384 ? 256 : ADV_THREADS;
    if (const char* v = getenv("DBAZ_ADV_THREADS")) { int x = atoi(v); if (x >= 32 && x <= ADV_THREADS && x % 32 == 0) e->adv_threads = x; }
    if (e->adv_smem > 48 * 1024) {
        cudaError_t s1 = cudaFuncSetAttribute(k_advance_roots<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->adv_smem);
        cudaError_t s2 = cudaFuncSetAttribute(k_advance_roots<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->adv_smem);
        if (s1 != cudaSuccess || s2 != cudaSuccess) { g_create_err = "cannot reserve shared memory for re-rooting"; dbaz_engine_destroy(e); return 1; }
    }
    k_build_act_tab<<<1, DBAZ_MAX_ACTIONS>>>(b, const_cast<uint4*>(ta.act_tab));
    cudaMemset(ta.pend, 0, (size_t)max_pending * ta.n_trees * 3 * sizeof(uint4));
    cudaMemset(ta.ctr, 0, 16 * sizeof(int));
    cudaMemset(ta.path_wn, 0, (size_t)ta.n_trees * PATH_CAP * sizeof(uint2));
    ta.batch_rows = 0x7fffffff;
    ta.phase = 0; ta.buf = 0;
    ta.cache_vcell = C;  // action C = horizontal edge (row 0, column C): always a padding cell
    cudaMemset(ta.path, 0, (size_t)max_pending * ta.n_trees * PATH_CAP * sizeof(uint32_t));
    // an all-empty-board root set so that the engine is usable right after create
    k_reset_roots<<<blocks_for(ta.n_trees, 128), 128>>>(b, ta, nullptr);
    if ((st = cudaDeviceSynchronize()) != cudaSuccess) { cuda_fail(nullptr, "k_reset_roots", st); dbaz_engine_destroy(e); return 1; }
    *out = e;
    return 0;
}

void dbaz_engine_destroy(dbaz_engine* e) {
    if (!e) return;
    DeviceGuard guard(e->cfg.device);
    cudaFree(e->ta.arena);
    cudaFree(e->ta.trees);
    cudaFree(e->ta.root_prior);
    cudaFree(e->ta.path);
    cudaFree(e->ta.path_wn);
    cudaFree(const_cast<double2*>(e->ta.lut));
    cudaFree(const_cast<uint4*>(e->ta.act_tab));
    cudaFree(e->ta.pend);
    cudaFree(e->ta.ctr);
    cudaFree(e->ta.cache);
    cudaFree(e->d_status);
    cudaFree(e->d_tower_err);
    cudaFree(e->d_cache_epoch);
    delete e;
}

int dbaz_engine_info(const dbaz_engine* e, int32_t* out8) {
    if (!e || !out8) return 1;
    out8[0] = e->board.L; out8[1] = e->board.C; out8[2] = e->board.A; out8[3] = e->board.F;
    out8[4] = e->ta.n_trees; out8[5] = e->ta.max_nodes; out8[6] = e->ta.stride; out8[7] = e->ta.max_pending;
    return 0;
}

int dbaz_engine_set_cpuct(dbaz_engine* e, double cpuct, double cpuct_base) {
    if (!e) return 1;
    if (cpuct == e->ta.cpuct && cpuct_base == e->ta.cpuct_base) return 0;
    DeviceGuard guard(e->cfg.device);
    DBAZ_CK(e, cudaDeviceSynchronize());
    e->ta.cpuct = cpuct; e->ta.cpuct_base = cpuct_base;
    e->cfg.cpuct = cpuct; e->cfg.cpuct_base = cpuct_base;
    return upload_lut(e);
}

/* ------------------------------------------------------------------ game */

int dbaz_game_init(dbaz_engine* e, dbaz_state* states, int64_t n, uint64_t stream) {
    if (!e) return 1;
    if (n <= 0) return 0;
    DeviceGuard guard(e->cfg.device);
    k_game_init<<<blocks_for(n, 256), 256, 0, S(stream)>>>(e->board, states, n);
    return launch_ok(e, "k_game_init");
}

int dbaz_game_valid_moves(dbaz_engine* e, const dbaz_state* states, uint8_t* out, int64_t n, uint64_t stream) {
    if (!e) return 1;
    if (n <= 0) return 0;
    DeviceGuard guard(e->cfg.device);
    if (e->nw == 1) k_game_valid<1><<<blocks_for(n, 256), 256, 0, S(stream)>>>(e->board, states, out, n);
    else k_game_valid<2><<<blocks_for(n, 256), 256, 0, S(stream)>>>(e->board, states, out, n);
    return launch_ok(e, "k_game_valid");
}

int dbaz_game_play(dbaz_engine* e, dbaz_state* states, const int32_t* moves, int32_t* n_closed, int32_t* closed_lc,
                   int64_t n, uint64_t stream) {
    if (!e) return 1;
    if (n <= 0) return 0;
    DeviceGuard guard(e->cfg.device);
    if (e->nw == 1) k_game_play<1><<<blocks_for(n, 256), 256, 0, S(stream)>>>(e->board, states, moves, n_closed, closed_lc, n);
    else k_game_play<2><<<blocks_for(n, 256), 256, 0, S(stream)>>>(e->board, states, moves, n_closed, closed_lc, n);
    return launch_ok(e, "k_game_play");
}

int dbaz_game_result(dbaz_engine* e, const dbaz_state* states, int8_t* out, int64_t n, uint64_t stream) {
    if (!e) return 1;
    if (n <= 0) return 0;
    DeviceGuard guard(e->cfg.device);
    k_game_result<<<blocks_for(n, 256), 256, 0, S(stream)>>>(states, out, n);
    return launch_ok(e, "k_game_result");
}

int dbaz_game_features(dbaz_engine* e, const dbaz_state* states, void* planes, int32_t dtype, int32_t layout, int64_t n,
                       uint64_t stream) {
    if (!e) return 1;
    if (dtype < DBAZ_F32 || dtype > DBAZ_I16 || layout < 0 || layout > 1) return fail(e, "bad dtype/layout");
    if (n <= 0) return 0;
    DeviceGuard guard(e->cfg.device);
    if (e->nw == 1) k_game_features<1><<<blocks_for(n * 32, 256), 256, 0, S(stream)>>>(e->board, states, planes, dtype, layout, n);
    else k_game_features<2><<<blocks_for(n * 32, 256), 256, 0, S(stream)>>>(e->board, states, planes, dtype, layout, n);
    return launch_ok(e, "k_game_features");
}

int dbaz_game_random_rollout(dbaz_engine* e, dbaz_state* states, uint64_t seed, uint64_t game0, int32_t* n_plies,
                             uint8_t* moves, int32_t max_plies, int64_t n, uint64_t stream) {
    if (!e) return 1;
    if (n <= 0) return 0;
    DeviceGuard guard(e->cfg.device);
    if (e->nw == 1) k_game_rollout<1><<<blocks_for(n, 128), 128, 0, S(stream)>>>(e->board, e->ta.act_tab, states, seed, game0, n_plies, moves, max_plies, n);
    else k_game_rollout<2><<<blocks_for(n, 128), 128, 0, S(stream)>>>(e->board, e->ta.act_tab, states, seed, game0, n_plies, moves, max_plies, n);
    return launch_ok(e, "k_game_rollout");
}

int dbaz_fake_nn(dbaz_engine* e, const dbaz_state* leaf_states, float* priors, float* values, int32_t kind, int64_t n,
                 uint64_t stream) {
    if (!e) return 1;
    if (n <= 0) return 0;
    DeviceGuard guard(e->cfg.device);
    k_fake_nn<<<blocks_for(n * 32, 256), 256, 0, S(stream)>>>(e->board, leaf_states, priors, values, kind, n);
    return launch_ok(e, "k_fake_nn");
}

/* ------------------------------------------------- leaf-eval fused stages */

int dbaz_nn_epilogue(dbaz_engine* e, void* x, const void* res, const float* bias, const float* scale, const float* shift,
                     int64_t rows, int32_t channels, int32_t dtype, int32_t mode, uint64_t stream) {
    if (!e || !x || !scale || !shift) return 1;
    if (mode < 0 || mode > 2) return fail(e, "bad epilogue mode");
    if (rows <= 0) return 0;
    DeviceGuard guard(e->cfg.device);
    const int per = dtype == DBAZ_F32 ? 4 : 8;
    if (dtype != DBAZ_F32 && dtype != DBAZ_BF16 && dtype != DBAZ_F16) return fail(e, "bad dtype");
    if (channels % per) return fail(e, "channels must be a multiple of the vector width");
    const int cv = channels / per;
    const int64_t n_vec64 = rows * cv;
    if (n_vec64 >= (int64_t)1 << 31) return fail(e, "epilogue tensor too large");
    const uint32_t n_vec = (uint32_t)n_vec64;
    // total threads must be a multiple of cv so that each thread owns a fixed channel group
    int block = 256;
    while (block % cv && block > 32) block >>= 1;
    int64_t want = std::min<int64_t>((n_vec + (int64_t)block * 4 - 1) / ((int64_t)block * 4), (int64_t)e->n_sms * 8);
    int grid = (int)std::max<int64_t>(want, 1);
    if ((int64_t)block % cv) {  // cv does not divide the block: make the grid supply the multiple
        int g = cv / std::__gcd(cv, block);
        grid = (grid + g - 1) / g * g;
    }
#define DBAZ_EPI(KERNEL, TYPE)                                                                                     \
    do {                                                                                                           \
        if (mode == 0) KERNEL<TYPE, 0><<<grid, block, 0, S(stream)>>>((TYPE*)x, (const TYPE*)res, bias, scale, shift, n_vec, channels); \
        else if (mode == 1) KERNEL<TYPE, 1><<<grid, block, 0, S(stream)>>>((TYPE*)x, (const TYPE*)res, bias, scale, shift, n_vec, channels); \
        else KERNEL<TYPE, 2><<<grid, block, 0, S(stream)>>>((TYPE*)x, (const TYPE*)res, bias, scale, shift, n_vec, channels); \
    } while (0)
    if (dtype == DBAZ_BF16) DBAZ_EPI(k_nn_epilogue16, __nv_bfloat16);
    else if (dtype == DBAZ_F16) DBAZ_EPI(k_nn_epilogue16, __half);
    else {
        if (mode == 0) k_nn_epilogue32<0><<<grid, block, 0, S(stream)>>>((float*)x, (const float*)res, bias, scale, shift, n_vec, channels);
        else if (mode == 1) k_nn_epilogue32<1><<<grid, block, 0, S(stream)>>>((float*)x, (const float*)res, bias, scale, shift, n_vec, channels);
        else k_nn_epilogue32<2><<<grid, block, 0, S(stream)>>>((float*)x, (const float*)res, bias, scale, shift, n_vec, channels);
    }
#undef DBAZ_EPI
    return launch_ok(e, "k_nn_epilogue");
}

int dbaz_nn_stem(dbaz_engine* e, const dbaz_state* leaf_states, const float* w01, const float* bias_pos, const float* k2_pos,
                 const float* scale, const float* shift, void* out, int32_t cout, int32_t dtype, int32_t mode, int64_t n,
                 uint64_t stream) {
    if (!e || !leaf_states || !w01 || !bias_pos || !k2_pos || !scale || !shift || !out) return 1;
    if (n <= 0) return 0;
    if (cout < 8 || cout > 256 || (cout & (cout - 1))) return fail(e, "dbaz_nn_stem: cout must be a power of two in [8, 256]");
    if (mode < 0 || mode > 1) return fail(e, "bad stem mode");
    DeviceGuard guard(e->cfg.device);
    if (dtype == DBAZ_BF16) return launch_stem<__nv_bfloat16>(e, leaf_states, w01, bias_pos, k2_pos, scale, shift, (__nv_bfloat16*)out, (int)n, cout, mode, S(stream));
    if (dtype == DBAZ_F16) return launch_stem<__half>(e, leaf_states, w01, bias_pos, k2_pos, scale, shift, (__half*)out, (int)n, cout, mode, S(stream));
    return fail(e, "dbaz_nn_stem: 16-bit output types only");
}

int dbaz_nn_stem_mma_pack(dbaz_engine* e, const void* w48, void* packed, int32_t cout, uint64_t stream) {
    if (!e || !w48 || !packed) return 1;
    if (cout < 64 || cout > 512 || cout % 64) return fail(e, "dbaz_nn_stem_mma_pack: cout must be a multiple of 64 in [64, 512]");
    DeviceGuard guard(e->cfg.device);
    const int n = (cout / 8) * 3 * 32;
    k_nn_stem_mma_pack<<<blocks_for(n, 256), 256, 0, S(stream)>>>((const uint16_t*)w48, (uint2*)packed, cout);
    return launch_ok(e, "k_nn_stem_mma_pack");
}

int dbaz_nn_stem_mma(dbaz_engine* e, const dbaz_state* leaf_states, const void* w48, void* out, int32_t cout, int32_t dtype,
                     int64_t n, uint64_t stream) {
    if (!e || !leaf_states || !w48 || !out) return 1;
    if (n <= 0) return 0;
    if (cout < 64 || cout > 512 || cout % 64) return fail(e, "dbaz_nn_stem_mma: cout must be a multiple of 64 in [64, 512]");
    if (n * e->board.rows * e->board.cols >= ((int64_t)1 << 31)) return fail(e, "dbaz_nn_stem_mma: too many rows");
    DeviceGuard guard(e->cfg.device);
    if (dtype == DBAZ_BF16) return launch_stem_mma<__nv_bfloat16>(e, leaf_states, (const __nv_bfloat16*)w48, (__nv_bfloat16*)out, n, cout, S(stream));
    if (dtype == DBAZ_F16) return launch_stem_mma<__half>(e, leaf_states, (const __half*)w48, (__half*)out, n, cout, S(stream));
    return fail(e, "dbaz_nn_stem_mma: 16-bit types only");
}

int dbaz_nn_stem_mma_tiles(dbaz_engine* e, const dbaz_state* leaf_states, const void* w48, void* tiles, int64_t n, uint64_t stream) {
    if (!e || !leaf_states || !w48 || !tiles) return 1;
    if (n <= 0) return 0;
    const TowerGeom g = tower_geom(e->board.rows, e->board.cols);
    if (!g.ok) return fail(e, "dbaz_nn_stem_mma_tiles: the tower kernel does not support this board");
    if (n * e->board.rows * e->board.cols >= ((int64_t)1 << 31)) return fail(e, "dbaz_nn_stem_mma_tiles: too many rows");
    DeviceGuard guard(e->cfg.device);
    return launch_stem_mma<__nv_bfloat16>(e, leaf_states, (const __nv_bfloat16*)w48, (__nv_bfloat16*)tiles, n, TOWER_C, S(stream),
                                          StemPlanar{g.nb, g.WP, g.plane, g.buf});
}

int dbaz_nn_heads(dbaz_engine* e, const void* logits, int32_t ld, int32_t dtype, float* priors, float* values, int64_t n,
                  uint64_t stream) {
    if (!e || !logits || !priors || !values) return 1;
    if (n <= 0) return 0;
    if (ld < e->board.A + 1) return fail(e, "dbaz_nn_heads: ld >= A + 1 (the value pre-activation is column A)");
    DeviceGuard guard(e->cfg.device);
    const int A = e->board.A;
    const int grid = blocks_for(n * 32, 256);
    if (dtype == DBAZ_BF16) k_nn_heads<__nv_bfloat16><<<grid, 256, 0, S(stream)>>>((const __nv_bfloat16*)logits, ld, A, priors, values, n);
    else if (dtype == DBAZ_F16) k_nn_heads<__half><<<grid, 256, 0, S(stream)>>>((const __half*)logits, ld, A, priors, values, n);
    else if (dtype == DBAZ_F32) k_nn_heads<float><<<grid, 256, 0, S(stream)>>>((const float*)logits, ld, A, priors, values, n);
    else return fail(e, "bad dtype");
    return launch_ok(e, "k_nn_heads");
}

int dbaz_nn_heads_mlp(dbaz_engine* e, const void* logits, int32_t ld, int32_t dtype, int32_t n_hidden, const float* v_w,
                      float* priors, float* values, int64_t n, uint64_t stream) {
    if (!e || !logits || !v_w || !priors || !values) return 1;
    if (n <= 0) return 0;
    if (n_hidden < 1 || n_hidden > 32 || ld < e->board.A + n_hidden) return fail(e, "dbaz_nn_heads_mlp: 1 <= n_hidden <= 32 and ld >= A + n_hidden");
    DeviceGuard guard(e->cfg.device);
    const int A = e->board.A;
    const int grid = blocks_for(n * 32, 256);
    if (dtype == DBAZ_BF16) k_nn_heads_mlp<__nv_bfloat16><<<grid, 256, 0, S(stream)>>>((const __nv_bfloat16*)logits, ld, A, n_hidden, v_w, priors, values, n);
    else if (dtype == DBAZ_F16) k_nn_heads_mlp<__half><<<grid, 256, 0, S(stream)>>>((const __half*)logits, ld, A, n_hidden, v_w, priors, values, n);
    else if (dtype == DBAZ_F32) k_nn_heads_mlp<float><<<grid, 256, 0, S(stream)>>>((const float*)logits, ld, A, n_hidden, v_w, priors, values, n);
    else return fail(e, "bad dtype");
    return launch_ok(e, "k_nn_heads_mlp");
}

/* ---------------------------------------------------------- residual tower */

int dbaz_nn_tower_geometry(dbaz_engine* e, int32_t* out8) {
    if (!e || !out8) return 1;
    const TowerGeom g = tower_geom(e->board.rows, e->board.cols);
    out8[0] = g.ok; out8[1] = g.nb; out8[2] = g.plane; out8[3] = g.buf; out8[4] = TOWER_CHUNK_BYTES;
    out8[5] = TOWER_CHUNKS_PER_STAGE; out8[6] = TOWER_C; out8[7] = g.WP;
    return 0;
}

int dbaz_nn_tower_planarize(dbaz_engine* e, const void* nhwc, void* tiles, int64_t n, uint64_t stream) {
    if (!e || !nhwc || !tiles) return 1;
    if (n <= 0) return 0;
    DeviceGuard guard(e->cfg.device);
    const std::string err = tower_planarize(tower_geom(e->board.rows, e->board.cols), nhwc, tiles, n, S(stream));
    return err.empty() ? 0 : fail(e, err);
}

int dbaz_nn_tower(dbaz_engine* e, const void* tiles, const void* packed_w, const float* bias, int32_t n_stages, int32_t head_cout,
                  void* out, int64_t n, uint64_t stream) {
    if (!e || !tiles || !packed_w || !bias || !out) return 1;
    if (n <= 0) return 0;
    DeviceGuard guard(e->cfg.device);
    if (!e->d_tower_err) {
        DBAZ_CK(e, cudaMalloc(&e->d_tower_err, sizeof(int)));
        DBAZ_CK(e, cudaMemset(e->d_tower_err, 0, sizeof(int)));
    }
    TowerLaunch a;
    a.blob = tiles; a.packed_w = packed_w; a.bias = bias; a.out = out; a.n_stages = n_stages; a.head_cout = head_cout;
    a.n_boards = n; a.n_sms = e->n_sms; a.err_flag = e->d_tower_err; a.dbg = e->tower_dbg;
    const std::string err = tower_launch(tower_geom(e->board.rows, e->board.cols), a, S(stream));
    return err.empty() ? 0 : fail(e, err);
}

int dbaz_nn_tower_trace(dbaz_engine* e, int64_t* timeline) {
    if (!e) return 1;
    e->tower_dbg = reinterpret_cast<long long*>(timeline);
    return 0;
}

/* ---------------------------------------------------------------- search */

int dbaz_search_reset_roots(dbaz_engine* e, const dbaz_state* root_states, uint64_t stream) {
    if (!e || !root_states) return 1;
    DeviceGuard guard(e->cfg.device);
    DBAZ_CK(e, cudaMemsetAsync(e->ta.ctr + 7, 0, sizeof(int), S(stream)));
    k_reset_roots<<<blocks_for(e->ta.n_trees, 128), 128, 0, S(stream)>>>(e->board, e->ta, root_states);
    e->noise = nullptr; e->coeff = 0.0;
    return launch_ok(e, "k_reset_roots");
}

int dbaz_search_begin(dbaz_engine* e, const int32_t* num_reads, int32_t pending, const double* noise, double coeff,
                      uint64_t stream) {
    if (!e || !num_reads) return 1;
    if (pending < 1 || pending > e->ta.max_pending) return fail(e, "pending must be in [1, max_pending of the engine]");
    DeviceGuard guard(e->cfg.device);
    e->noise = noise; e->coeff = coeff; e->pending = pending;
    DBAZ_CK(e, cudaMemsetAsync(e->ta.ctr + 4, 0, 2 * sizeof(int), S(stream)));  // k_search_begin counts the busy trees into ctr[5]
    const int grid = blocks_for(e->ta.n_trees, TREE_WARPS);
    DBAZ_DISPATCH(e, (k_search_begin<APL, NW><<<grid, TREE_WARPS * 32, 0, S(stream)>>>(e->board, e->ta, num_reads, noise, coeff)));
    return launch_ok(e, "k_search_begin");
}

int dbaz_search_step(dbaz_engine* e, const float* priors, const float* values, void* planes, int32_t dtype, int32_t layout,
                     dbaz_state* leaf_states, int8_t* leaf_kind, uint64_t stream) {
    if (!e || !priors || !values || !planes) return 1;
    if (dtype < DBAZ_F32 || dtype > DBAZ_I16 || layout < 0 || layout > 1) return fail(e, "bad dtype/layout");
    DeviceGuard guard(e->cfg.device);
    const int grid = blocks_for(e->ta.n_trees, TREE_WARPS);
    if (e->pending == 1)
        DBAZ_DISPATCH(e, (k_search_step<APL, NW, true><<<grid, TREE_WARPS * 32, 0, S(stream)>>>(
                             e->board, e->ta, 1, priors, values, e->noise, e->coeff, planes, dtype, layout, leaf_states, leaf_kind)));
    else
        DBAZ_DISPATCH(e, (k_search_step<APL, NW, false><<<grid, TREE_WARPS * 32, 0, S(stream)>>>(
                             e->board, e->ta, e->pending, priors, values, e->noise, e->coeff, planes, dtype, layout, leaf_states, leaf_kind)));
    return launch_ok(e, "k_search_step");
}

int dbaz_search_step2(dbaz_engine* e, int32_t phase, int32_t buf, int32_t max_inline, const float* priors, const float* values, void* planes,
                      int32_t dtype, int32_t layout, dbaz_state* leaf_states, uint64_t stream) {
    if (!e || !planes || !leaf_states) return 1;
    if (phase != 1 && phase != 2) return fail(e, "dbaz_search_step2: phase must be 1 (absorb) or 2 (chain)");
    if (phase == 1 && (!priors || !values)) return 1;
    if (buf < 0 || buf > 1 || max_inline < 0) return fail(e, "dbaz_search_step2: bad batch index / max_inline");
    if (e->pending != 1 || !e->ta.compact) return fail(e, "dbaz_search_step2 needs max_pending_evals == 1 and compact rows (dbaz_search_set_mode)");
    if (dtype < DBAZ_F32 || dtype > DBAZ_I16 || layout < 0 || layout > 1) return fail(e, "bad dtype/layout");
    DeviceGuard guard(e->cfg.device);
    TreeArgs ta = e->ta;
    ta.phase = phase; ta.buf = buf; ta.max_inline = max_inline;
    const int grid = blocks_for(ta.n_trees, TREE_WARPS);
    DBAZ_DISPATCH(e, (k_search_step<APL, NW, true><<<grid, TREE_WARPS * 32, 0, S(stream)>>>(
                         e->board, ta, 1, priors, values, e->noise, e->coeff, planes, dtype, layout, leaf_states, nullptr)));
    return launch_ok(e, "k_search_step (phase)");
}

/* ---------------------------------------------------------- one graph per search */

struct dbaz_loop {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    LoopCtl* d_ctl = nullptr;
    int n_rungs = 0;
};

int dbaz_search_loop_build(dbaz_engine* e, const uint64_t* rung_graphs, const int32_t* rung_rows, const float* rung_us, int32_t n_rungs,
                           int32_t max_iters, float row_margin, float undersize, float undersize_gain, float wave_overhead_us,
                           uint64_t* loop_out) {
    if (!e || !rung_graphs || !rung_rows || !rung_us || !loop_out) return 1;
    if (n_rungs < 1 || n_rungs > LOOP_MAX_RUNGS) return fail(e, "dbaz_search_loop_build: 1..48 rungs");
    for (int r = 1; r < n_rungs; ++r)
        if (rung_rows[r] >= rung_rows[r - 1]) return fail(e, "dbaz_search_loop_build: rung rows must be strictly descending");
    DeviceGuard guard(e->cfg.device);
    dbaz_loop* L = new dbaz_loop();
    L->n_rungs = n_rungs;
    LoopCtl h;
    memset(&h, 0, sizeof h);
    h.n_rungs = n_rungs;
    for (int r = 0; r < n_rungs; ++r) { h.rows[r] = rung_rows[r]; h.us[r] = rung_us[r]; }
    h.row_margin = row_margin; h.undersize = undersize; h.undersize_gain = undersize_gain; h.wave_overhead_us = wave_overhead_us;
    h.max_iters = max_iters > 0 ? max_iters : 1;
#define LOOP_CK(call)                                                                   \
    do {                                                                                \
        cudaError_t st_ = (call);                                                       \
        if (st_ != cudaSuccess) {                                                       \
            if (L->exec) cudaGraphExecDestroy(L->exec);                                 \
            if (L->graph) cudaGraphDestroy(L->graph);                                   \
            cudaFree(L->d_ctl);                                                         \
            delete L;                                                                   \
            return cuda_fail(e, #call, st_);                                            \
        }                                                                               \
    } while (0)
    LOOP_CK(cudaMalloc(&L->d_ctl, sizeof(LoopCtl)));
    LOOP_CK(cudaMemcpy(L->d_ctl, &h, sizeof h, cudaMemcpyHostToDevice));
    LOOP_CK(cudaGraphCreate(&L->graph, 0));
    cudaGraphConditionalHandle h_while, h_switch;
    LOOP_CK(cudaGraphConditionalHandleCreate(&h_while, L->graph, 0, 0));
    LOOP_CK(cudaGraphConditionalHandleCreate(&h_switch, L->graph, 0, 0));
    int* ctr = e->ta.ctr;
    void* args[4] = {&ctr, &L->d_ctl, &h_while, &h_switch};
    cudaKernelNodeParams kp;
    memset(&kp, 0, sizeof kp);
    kp.gridDim = dim3(1); kp.blockDim = dim3(32); kp.sharedMemBytes = 0; kp.kernelParams = args; kp.extra = nullptr;
    // begin kernel
    cudaGraphNode_t n_begin;
    kp.func = (void*)k_loop_begin;
    LOOP_CK(cudaGraphAddKernelNode(&n_begin, L->graph, nullptr, 0, &kp));
    // WHILE node
    cudaGraphNodeParams wp = {cudaGraphNodeTypeConditional};
    wp.type = cudaGraphNodeTypeConditional;
    wp.conditional.handle = h_while;
    wp.conditional.type = cudaGraphCondTypeWhile;
    wp.conditional.size = 1;
    cudaGraphNode_t n_while;
    LOOP_CK(cudaGraphAddNode(&n_while, L->graph, &n_begin, 1, &wp));
    cudaGraph_t body = wp.conditional.phGraph_out[0];
    // SWITCH node inside the body
    cudaGraphNodeParams sp = {cudaGraphNodeTypeConditional};
    sp.type = cudaGraphNodeTypeConditional;
    sp.conditional.handle = h_switch;
    sp.conditional.type = cudaGraphCondTypeSwitch;
    sp.conditional.size = (unsigned)n_rungs;
    cudaGraphNode_t n_switch;
    LOOP_CK(cudaGraphAddNode(&n_switch, body, nullptr, 0, &sp));
    for (int r = 0; r < n_rungs; ++r) {
        cudaGraphNode_t child;
        LOOP_CK(cudaGraphAddChildGraphNode(&child, sp.conditional.phGraph_out[r], nullptr, 0, reinterpret_cast<cudaGraph_t>(rung_graphs[r])));
    }
    // decide kernel after the switch
    cudaGraphNode_t n_decide;
    kp.func = (void*)k_loop_decide;
    LOOP_CK(cudaGraphAddKernelNode(&n_decide, body, &n_switch, 1, &kp));
    LOOP_CK(cudaGraphInstantiate(&L->exec, L->graph, 0));
#undef LOOP_CK
    *loop_out = reinterpret_cast<uint64_t>(L);
    return 0;
}

int dbaz_search_loop_pick(const int32_t* rung_rows, const float* rung_us, int32_t n_rungs, float undersize, float undersize_gain,
                          float wave_overhead_us, int32_t want) {
    if (!rung_rows || !rung_us || n_rungs < 1 || n_rungs > LOOP_MAX_RUNGS) return -1;
    LoopCtl c;
    memset(&c, 0, sizeof c);
    c.n_rungs = n_rungs;
    for (int r = 0; r < n_rungs; ++r) { c.rows[r] = rung_rows[r]; c.us[r] = rung_us[r]; }
    c.undersize = undersize; c.undersize_gain = undersize_gain; c.wave_overhead_us = wave_overhead_us;
    return loop_pick(&c, want);
}

int dbaz_search_loop_launch(dbaz_engine* e, uint64_t loop, uint64_t stream) {
    if (!e || !loop) return 1;
    dbaz_loop* L = reinterpret_cast<dbaz_loop*>(loop);
    DeviceGuard guard(e->cfg.device);
    DBAZ_CK(e, cudaGraphLaunch(L->exec, S(stream)));
    return 0;
}

int dbaz_search_loop_counts(dbaz_engine* e, uint64_t loop, uint32_t* replays_out, uint64_t stream) {
    if (!e || !loop || !replays_out) return 1;
    dbaz_loop* L = reinterpret_cast<dbaz_loop*>(loop);
    DeviceGuard guard(e->cfg.device);
    // copy the per-rung replay counts out and zero them, in stream order
    DBAZ_CK(e, cudaMemcpyAsync(replays_out, L->d_ctl->replays, (size_t)L->n_rungs * sizeof(uint32_t), cudaMemcpyDefault, S(stream)));
    DBAZ_CK(e, cudaMemsetAsync(L->d_ctl->replays, 0, (size_t)L->n_rungs * sizeof(uint32_t), S(stream)));
    return 0;
}

void dbaz_search_loop_destroy(dbaz_engine* e, uint64_t loop) {
    if (!loop) return;
    dbaz_loop* L = reinterpret_cast<dbaz_loop*>(loop);
    if (e) cudaSetDevice(e->cfg.device);
    if (L->exec) cudaGraphExecDestroy(L->exec);
    if (L->graph) cudaGraphDestroy(L->graph);
    cudaFree(L->d_ctl);
    delete L;
}

int dbaz_search_stop(dbaz_engine* e, uint64_t stream) {
    if (!e) return 1;
    DeviceGuard guard(e->cfg.device);
    k_search_stop<<<blocks_for(e->ta.n_trees, 128), 128, 0, S(stream)>>>(e->ta);
    return launch_ok(e, "k_search_stop");
}

int dbaz_search_root_visits(dbaz_engine* e, int32_t* out, uint64_t stream) {
    if (!e || !out) return 1;
    DeviceGuard guard(e->cfg.device);
    k_root_visits<<<blocks_for((int64_t)e->ta.n_trees * 32, 256), 256, 0, S(stream)>>>(e->board, e->ta, out);
    return launch_ok(e, "k_root_visits");
}

int dbaz_search_root_children(dbaz_engine* e, float* W, double* priors, int32_t* sign, double* ucb, uint64_t stream) {
    if (!e) return 1;
    DeviceGuard guard(e->cfg.device);
    const int grid = blocks_for((int64_t)e->ta.n_trees * 32, 256);
    if (e->nw == 1) k_root_children<1><<<grid, 256, 0, S(stream)>>>(e->board, e->ta, W, priors, sign, ucb);
    else k_root_children<2><<<grid, 256, 0, S(stream)>>>(e->board, e->ta, W, priors, sign, ucb);
    return launch_ok(e, "k_root_children");
}

int dbaz_search_node(dbaz_engine* e, int32_t tree, int32_t node, dbaz_state* state_out, float* W, int32_t* N, double* priors,
                     int32_t* child, int32_t* sign, double* ucb, int32_t* own8, float* own_W, uint64_t stream) {
    if (!e || !state_out || !W || !N || !priors || !child || !sign || !ucb || !own8 || !own_W) return 1;
    if (tree < 0 || tree >= e->ta.n_trees) return fail(e, "dbaz_search_node: no such tree");
    DeviceGuard guard(e->cfg.device);
    if (e->nw == 1) k_node_view<1><<<1, 32, 0, S(stream)>>>(e->board, e->ta, tree, node, state_out, W, N, priors, child, sign, ucb, own8, own_W);
    else k_node_view<2><<<1, 32, 0, S(stream)>>>(e->board, e->ta, tree, node, state_out, W, N, priors, child, sign, ucb, own8, own_W);
    return launch_ok(e, "k_node_view");
}

int dbaz_search_tree_stats(dbaz_engine* e, int32_t* stats8, float* root_W, float* q, uint64_t stream) {
    if (!e) return 1;
    DeviceGuard guard(e->cfg.device);
    k_tree_stats<<<blocks_for(e->ta.n_trees, 128), 128, 0, S(stream)>>>(e->ta, stats8, root_W, q);
    return launch_ok(e, "k_tree_stats");
}

int dbaz_search_tree_busy(dbaz_engine* e, int8_t* out, uint64_t stream) {
    if (!e || !out) return 1;
    DeviceGuard guard(e->cfg.device);
    k_tree_busy<<<blocks_for(e->ta.n_trees, 256), 256, 0, S(stream)>>>(e->ta, out);
    return launch_ok(e, "k_tree_busy");
}

int dbaz_search_root_states(dbaz_engine* e, dbaz_state* out, uint64_t stream) {
    if (!e || !out) return 1;
    DeviceGuard guard(e->cfg.device);
    k_root_states<<<blocks_for(e->ta.n_trees, 128), 128, 0, S(stream)>>>(e->ta, out);
    return launch_ok(e, "k_root_states");
}

int dbaz_search_advance_roots(dbaz_engine* e, const int32_t* moves, int32_t reuse, uint64_t stream) {
    if (!e || !moves) return 1;
    DeviceGuard guard(e->cfg.device);
    if (e->nw == 1) k_advance_roots<1><<<e->ta.n_trees, e->adv_threads, e->adv_smem, S(stream)>>>(e->board, e->ta, moves, reuse);
    else k_advance_roots<2><<<e->ta.n_trees, e->adv_threads, e->adv_smem, S(stream)>>>(e->board, e->ta, moves, reuse);
    e->noise = nullptr; e->coeff = 0.0;
    return launch_ok(e, "k_advance_roots");
}

static int selfplay_args(dbaz_engine* e, const dbaz_selfplay_buffers* b, SelfplayArgs& sp) {
    if (!b->inv_temp || !b->uniforms || !b->reads_by_k || !b->searching || !b->move_idx || !b->moves || !b->h_states || !b->h_visits ||
        !b->h_active || !b->h_moves || !b->h_stats || !b->h_q || !b->reads || !b->left || b->n_moves <= 0 || (b->noise && !b->noise_buf))
        return fail(e, "dbaz_selfplay: a required buffer is NULL or n_moves <= 0");
    sp.n_moves = b->n_moves; sp.inv_temp = b->inv_temp; sp.uniforms = b->uniforms; sp.noise = b->noise; sp.reads_by_k = b->reads_by_k;
    sp.searching = b->searching; sp.move_idx = b->move_idx; sp.moves = b->moves; sp.h_states = b->h_states; sp.h_visits = b->h_visits;
    sp.h_active = b->h_active; sp.h_moves = b->h_moves; sp.h_stats = b->h_stats; sp.h_q = b->h_q; sp.noise_buf = b->noise_buf;
    sp.reads = b->reads; sp.left = b->left;
    return 0;
}

int dbaz_selfplay_pick(dbaz_engine* e, const dbaz_selfplay_buffers* bufs, uint64_t stream) {
    if (!e || !bufs) return 1;
    SelfplayArgs sp;
    if (int rc = selfplay_args(e, bufs, sp)) return rc;
    DeviceGuard guard(e->cfg.device);
    k_selfplay_pick<<<blocks_for(e->ta.n_trees, SP_WARPS), SP_WARPS * 32, 0, S(stream)>>>(e->board, e->ta, sp);
    return launch_ok(e, "k_selfplay_pick");
}

int dbaz_selfplay_restart(dbaz_engine* e, const dbaz_selfplay_buffers* bufs, int32_t first, uint64_t stream) {
    if (!e || !bufs) return 1;
    SelfplayArgs sp;
    if (int rc = selfplay_args(e, bufs, sp)) return rc;
    DeviceGuard guard(e->cfg.device);
    if (e->nw == 1) k_selfplay_restart<1><<<blocks_for(e->ta.n_trees, SP_WARPS), SP_WARPS * 32, 0, S(stream)>>>(e->board, e->ta, sp, first);
    else k_selfplay_restart<2><<<blocks_for(e->ta.n_trees, SP_WARPS), SP_WARPS * 32, 0, S(stream)>>>(e->board, e->ta, sp, first);
    return launch_ok(e, "k_selfplay_restart");
}

int dbaz_search_set_chain_budget(dbaz_engine* e, int32_t microseconds) {
    if (!e) return 1;
    if (microseconds < 0 || microseconds > 100000) return fail(e, "chain budget must be in [0, 100000] microseconds");
    int khz = 0;
    DBAZ_CK(e, cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, e->cfg.device));
    e->ta.chain_clk = (int)std::min<long long>(0x7fffffffll, (long long)microseconds * (long long)khz / 1000ll);
    return 0;
}

int dbaz_search_set_mode(dbaz_engine* e, int32_t compact, int32_t max_inline) {
    if (!e) return 1;
    if (max_inline < 0) return fail(e, "max_inline must be >= 0");
    e->ta.compact = compact ? 1 : 0;
    e->ta.max_inline = max_inline;
    return 0;
}

int dbaz_search_set_batch_rows(dbaz_engine* e, int32_t rows) {
    if (!e) return 1;
    if (rows < 0) return fail(e, "rows must be >= 0");
    e->ta.batch_rows = rows > 0 ? rows : 0x7fffffff;
    return 0;
}

int dbaz_search_wave_counts(dbaz_engine* e, int32_t* out4, uint64_t stream) {
    if (!e || !out4) return 1;
    DeviceGuard guard(e->cfg.device);
    DBAZ_CK(e, cudaMemcpyAsync(out4, e->ta.ctr + 4, 4 * sizeof(int), cudaMemcpyDefault, S(stream)));
    DBAZ_CK(e, cudaMemsetAsync(e->ta.ctr + 6, 0, sizeof(int), S(stream)));  // the maximum restarts with every read
    return 0;
}

int dbaz_cache_configure(dbaz_engine* e, int32_t log2_entries) {
    if (!e) return 1;
    if (log2_entries < 0 || log2_entries > 30) return fail(e, "log2_entries must be in [0, 30]");
    DeviceGuard guard(e->cfg.device);
    DBAZ_CK(e, cudaDeviceSynchronize());
    if (e->ta.cache) { cudaFree(e->ta.cache); e->ta.cache = nullptr; }
    e->ta.cache_mask = 0; e->cache_log2 = 0;
    if (log2_entries == 0) return 0;
    const size_t bytes = ((size_t)1 << log2_entries) * (size_t)e->board.A * sizeof(uint4);
    cudaError_t st = cudaMalloc((void**)&e->ta.cache, bytes);
    if (st != cudaSuccess) {
        e->ta.cache = nullptr;
        char buf[160];
        std::snprintf(buf, sizeof buf, "cudaMalloc(eval cache, %zu bytes): %s", bytes, cudaGetErrorString(st));
        return fail(e, buf);
    }
    e->ta.cache_mask = (uint32_t)(((size_t)1 << log2_entries) - 1);
    e->cache_log2 = log2_entries;
    DBAZ_CK(e, cudaMemset(e->ta.cache, 0xff, bytes));  // all-ones edges never occur (padding bits stay clear)
    if (!e->d_cache_epoch) DBAZ_CK(e, cudaMalloc(&e->d_cache_epoch, sizeof(uint32_t)));
    e->cache_epoch = 1;
    DBAZ_CK(e, cudaMemcpy(e->d_cache_epoch, &e->cache_epoch, sizeof(uint32_t), cudaMemcpyHostToDevice));
    e->ta.cache_epoch = e->d_cache_epoch;
    return 0;
}

int dbaz_cache_clear(dbaz_engine* e, uint64_t stream) {
    if (!e) return 1;
    if (!e->ta.cache) return 0;
    DeviceGuard guard(e->cfg.device);
    // every key carries the table epoch: a new epoch makes every stored entry a miss.  Only when the 32-bit epoch is about
    // to run out is the table really wiped (8.6 GB at 2^24 entries of a 3x3 board: ~2.5 ms that a step does not have)
    if (e->cache_epoch >= 0xfffffff0u) {
        const size_t bytes = ((size_t)e->ta.cache_mask + 1) * (size_t)e->board.A * sizeof(uint4);
        DBAZ_CK(e, cudaMemsetAsync(e->ta.cache, 0xff, bytes, S(stream)));
        e->cache_epoch = 0;
    }
    e->cache_epoch += 1;
    k_cache_epoch<<<1, 1, 0, S(stream)>>>(e->d_cache_epoch, e->cache_epoch);
    return launch_ok(e, "k_cache_epoch");
}

int dbaz_search_status(dbaz_engine* e, int64_t* out8, uint64_t stream) {
    if (!e) return 1;
    DeviceGuard guard(e->cfg.device);
    DBAZ_CK(e, cudaMemsetAsync(e->d_status, 0, 8 * sizeof(unsigned long long), S(stream)));
    k_status<<<blocks_for(e->ta.n_trees, 128), 128, 0, S(stream)>>>(e->ta, e->d_status);
    if (launch_ok(e, "k_status")) return 1;
    unsigned long long h[8];
    DBAZ_CK(e, cudaMemcpyAsync(h, e->d_status, sizeof h, cudaMemcpyDeviceToHost, S(stream)));
    DBAZ_CK(e, cudaStreamSynchronize(S(stream)));
    if (out8) for (int i = 0; i < 8; ++i) out8[i] = (int64_t)h[i];
    if (h[0]) {
        char buf[160];
        std::snprintf(buf, sizeof buf, "%llu tree(s) faulted: node pool exhausted (max_nodes=%d) or illegal re-root move",
                      h[0], e->ta.max_nodes);
        return fail(e, buf);
    }
    return 0;
}

}  // extern "C"
