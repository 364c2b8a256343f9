// dbaz_trunk.cu -- one 256 -> 256 channel 3x3 convolution of SimpleNN's trunk (dots_boxes_nn.py; FusedSimpleNN runs conv1-conv3 here) as a
// persistent sm_100a GEMM per output position that multiplies only the taps inside the board.
//
// Why.  On the 4 x 4 points of a 3 x 3 board only 100 of the 144 taps of a padded 3x3 convolution fall inside the board;
// an implicit GEMM with K = 9 x 256 multiplies the other 31 % by zeros.  Here a work item is (128 boards, ONE output
// position p): a GEMM with M = 128 boards, N = 256 output channels and K = taps(p) x 256, whose K loop walks the in-board
// taps of p only.  Its accumulator (128 lanes x 256 fp32 columns) is half of tensor memory, so two accumulators let the
// epilogue drain item i while the MMAs of item i + 1 run.
//
//   y[b, p, :] = relu( (sum over in-board taps t of p:  x[b, q_t, :] . W_t  +  bias_pos[p, :])  +  bias[:] )
//
// * K step = (64 input channels, tap): TMA loads the 128 boards' 128-byte channel slice at input position q_t (A, 16 KB)
//   and tap t's [256 cout][64 cin] weight slice (B, 32 KB), both in the 128-byte swizzle; four K = 16 MMAs per step.
//   Operand traffic is 48 KB per 4.2 MFLOP, the same ratio as cuDNN's 256 x 128 CTA-pair tile.
// * Every output element accumulates in one fixed order -- 64-channel chunks ascending, inside a chunk the taps by
//   (ky, kx) -- whatever n, the row a board sits in or the CTA that runs the item: a board's output is a function of its
//   own input alone.  It is the order of cuDNN's implicit GEMM for this conv (NHWC, K = (ky, kx, c)); a padding tap
//   only adds exact zeros there, and with the same bf16-rounded biases added in the same order, the output equals the
//   library's conv-add-bias-ReLU (z = bias_pos) bit for bit (tests/test_gpu_trunk_conv.py).
// * Items are handed out by descending tap count (9, 6, 4 on 3 x 3) in a snake over the persistent CTAs, so each CTA gets
//   a similar amount of work and the grid ends on the cheap corner items; beyond 4096 boards, in chunks of 4096 boards
//   whose activations stay in L2 while all their positions are computed.
// * Rows >= n of the output are never written (rows >= n of the input are read and computed: M rows are independent).
// * Warp roles: 0 TMA producer, 1 MMA issuer (owns the tensor memory), 2..5 epilogue (tcgen05.ld -> + bias_pos in fp32 ->
//   ReLU in the bf16 conversion -> 512 contiguous bytes per board to global memory).  Every mbarrier wait is bounded.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <string.h>
#include <string>

#include "dbaz_tcgen05.cuh"
#include "dbaz_trunk.cuh"

namespace dbaz {

namespace {

constexpr int TK_WARPS = 6;
constexpr int TK_THREADS = TK_WARPS * 32;
constexpr int TK_NS = 4;                                   // pipeline stages
constexpr uint32_t TK_A_BYTES = TRUNK_BM * 128;            // 128 boards x 64 channels bf16
constexpr uint32_t TK_B_BYTES = TRUNK_C * 128;             // 256 output channels x 64 input channels bf16
constexpr uint32_t TK_STAGE = TK_A_BYTES + TK_B_BYTES;
constexpr uint32_t TK_TMEM_COLS = 512;                     // two accumulators of 256 columns
constexpr size_t TK_SMEM = 1024 + TK_NS * (size_t)TK_STAGE + 256;
constexpr int TK_MAGIC = 0x7472756b;

constexpr int TK_CHUNK = 32;                               // tiles per chunk of the item order (4096 boards)

// work item of round r of this CTA (snake over the grid), -1 past the end
__device__ __forceinline__ int trunk_item(int r, int n_items) {
    const int G = (int)gridDim.x, b = (int)blockIdx.x;
    const int i = r * G + ((r & 1) ? G - 1 - b : b);
    return i < n_items ? i : -1;
}
// Item -> (output position, tile).  Items run in chunks of TK_CHUNK tiles, by descending tap count inside a chunk: the
// chunk's activations (8 KB per board on 4 x 4) stay in L2 while its positions read each of them several times.  With at
// most TK_CHUNK tiles this is simply rank-major.
__device__ __forceinline__ void trunk_decode(const TrunkParams& P, int item, int& p, int& tile) {
    const int per = TK_CHUNK * P.taps.n_out;
    const int c = item / per, r = item - c * per;
    const int tc = min(TK_CHUNK, P.n_tiles - c * TK_CHUNK);
    p = P.taps.order[r / tc];
    tile = c * TK_CHUNK + r % tc;
}

__global__ void __launch_bounds__(TK_THREADS, 1)
k_trunk_conv(const __grid_constant__ CUtensorMap amap, const __grid_constant__ CUtensorMap wmap, const __grid_constant__ TrunkParams P) {
    extern __shared__ unsigned char smem_dyn[];
    const uint32_t raw = smem_u32(smem_dyn);
    const uint32_t base = (raw + 1023u) & ~1023u;          // the 128-byte swizzle wants 1024-byte aligned tiles
    const uint32_t BAR = base + TK_NS * TK_STAGE;
    const uint32_t full = BAR, empty = BAR + 8 * TK_NS, acc_full = BAR + 16 * TK_NS, acc_empty = acc_full + 16,
                   tmem_slot = acc_empty + 16;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int i = 0; i < TK_NS; ++i) { mbar_init(full + 8 * i, 1); mbar_init(empty + 8 * i, 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(acc_full + 8 * i, 1); mbar_init(acc_empty + 8 * i, 128); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TK_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(tmem_slot));

    const int n_items = P.n_items;

    if (warp == 0) {
        // =================== TMA producer: one thread streams (A, B) per K step
        if (lane == 0) {
            uint32_t s = 0;
            for (int r = 0;; ++r) {
                const int item = trunk_item(r, n_items);
                if (item < 0) break;
                int p, tile;
                trunk_decode(P, item, p, tile);
                const int cnt = P.taps.count[p];
                for (int j = 0; j < 4 * cnt; ++j, ++s) {
                    const int k = j % cnt, c = j / cnt;  // channel chunk outer, tap inner: cuDNN's order of K
                    const int e = P.taps.tap[p][k], t = e & 15, q = e >> 4;
                    {
                        const uint32_t slot = s % TK_NS, ph = (s / TK_NS) & 1u;
                        mbar_wait(empty + 8 * slot, ph ^ 1u, P.err, 1);
                        const uint32_t a = base + slot * TK_STAGE, b = a + TK_A_BYTES;
                        mbar_expect_tx(full + 8 * slot, TK_STAGE);
                        tma_load_3d(a, &amap, 64 * c, q, TRUNK_BM * tile, full + 8 * slot);
                        tma_load_2d(b, &wmap, 64 * c, TRUNK_C * t, full + 8 * slot);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // =================== MMA issuer: the whole warp runs the loop, one elected lane issues and commits
        const uint32_t idesc = umma_idesc(TRUNK_C);
        uint32_t s = 0, a = 0;
        for (int r = 0;; ++r, ++a) {
            const int item = trunk_item(r, n_items);
            if (item < 0) break;
            int p, tile;
            trunk_decode(P, item, p, tile);
            const int steps = 4 * P.taps.count[p];
            const uint32_t acc = a & 1u;
            mbar_wait(acc_empty + 8 * acc, ((a >> 1) & 1u) ^ 1u, P.err, 2);
            tc_fence_after();
            const uint32_t d = tmem + acc * TRUNK_C;
            for (int j = 0; j < steps; ++j, ++s) {
                const uint32_t slot = s % TK_NS, ph = (s / TK_NS) & 1u;
                mbar_wait(full + 8 * slot, ph, P.err, 3);
                tc_fence_after();
                const uint32_t a_lo = (((base + slot * TK_STAGE) >> 4) & 0x3fffu) | (1u << 16);
                const uint32_t b_lo = (((base + slot * TK_STAGE + TK_A_BYTES) >> 4) & 0x3fffu) | (1u << 16);
                if (elect_one()) {
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        umma(d, desc64_sw128(a_lo + 2u * kk), desc64_sw128(b_lo + 2u * kk), idesc, (j | kk) != 0 ? 1u : 0u);
                    umma_commit(empty + 8 * slot);
                }
                __syncwarp();
            }
            if (elect_one()) umma_commit(acc_full + 8 * acc);
            __syncwarp();
        }
    } else {
        // =================== epilogue: warp w reads accumulator lanes 32 (w % 4) .. +31, i.e. boards 32 (w % 4) + lane
        const int quad = warp & 3, row = 32 * quad + lane;
        const int n_out = P.taps.n_out;
        uint32_t a = 0;
        for (int r = 0;; ++r, ++a) {
            const int item = trunk_item(r, n_items);
            if (item < 0) break;
            int p, tile;
            trunk_decode(P, item, p, tile);
            const int64_t board = (int64_t)TRUNK_BM * tile + row;
            const bool ok = board < P.n;
            const uint32_t acc = a & 1u;
            mbar_wait(acc_full + 8 * acc, (a >> 1) & 1u, P.err, 4);
            tc_fence_after();
            const float4* bp = reinterpret_cast<const float4*>(P.bias_pos + (size_t)p * TRUNK_C);
            const float4* bc = reinterpret_cast<const float4*>(P.bias);
            uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(P.out) + ((size_t)board * n_out + p) * TRUNK_C);
#pragma unroll 1
            for (int j = 0; j < TRUNK_C / 32; ++j) {
                uint32_t v[32];
                tmem_ld32(tmem + ((uint32_t)(32 * quad) << 16) + acc * TRUNK_C + 32u * j, v);
                float z[32], b[32];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float4 f = __ldg(bp + 8 * j + i), g = __ldg(bc + 8 * j + i);
                    z[4 * i] = f.x; z[4 * i + 1] = f.y; z[4 * i + 2] = f.z; z[4 * i + 3] = f.w;
                    b[4 * i] = g.x; b[4 * i + 1] = g.y; b[4 * i + 2] = g.z; b[4 * i + 3] = g.w;
                }
                tmem_ld_wait();
                float f[32];
#pragma unroll
                for (int i = 0; i < 32; ++i)
                    f[i] = __fadd_rn(__fadd_rn(__uint_as_float(v[i]), z[i]), b[i]);
                uint32_t o[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) o[i] = pack_relu_bf16(f[2 * i], f[2 * i + 1]);
                if (ok) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) op[4 * j + c] = make_uint4(o[4 * c], o[4 * c + 1], o[4 * c + 2], o[4 * c + 3]);
                }
            }
            tc_fence_before();
            mbar_arrive(acc_empty + 8 * acc);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TK_TMEM_COLS) : "memory");
    }
}

}  // namespace

std::string trunk_taps(int hi, int wi, int pad, TrunkTaps* t) {
    if (pad != 0 && pad != 1) return "trunk conv: pad must be 0 or 1";
    const int ho = hi + 2 * pad - 2, wo = wi + 2 * pad - 2;
    if (hi < 1 || wi < 1 || ho < 1 || wo < 1) return "trunk conv: the grid is smaller than the kernel";
    if (hi * wi > TRUNK_MAX_POS) return "trunk conv: more than 64 input positions";
    memset(t, 0, sizeof(*t));
    t->hi = hi; t->wi = wi; t->pad = pad; t->ho = ho; t->wo = wo; t->n_out = ho * wo;
    for (int y = 0; y < ho; ++y)
        for (int x = 0; x < wo; ++x) {
            const int p = y * wo + x;
            int k = 0;
            for (int ky = 0; ky < 3; ++ky)
                for (int kx = 0; kx < 3; ++kx) {
                    const int iy = y + ky - pad, ix = x + kx - pad;
                    if (iy < 0 || iy >= hi || ix < 0 || ix >= wi) continue;
                    t->tap[p][k++] = (uint16_t)(((iy * wi + ix) << 4) | (3 * ky + kx));
                }
            t->count[p] = (uint8_t)k;
        }
    int r = 0;
    for (int c = 9; c >= 1; --c)
        for (int p = 0; p < t->n_out; ++p)
            if (t->count[p] == c) t->order[r++] = (uint8_t)p;
    return "";
}

std::string trunk_plan(const TrunkPlanArgs& a, TrunkPlan* plan) {
    memset(plan, 0, sizeof(*plan));
    std::string err = trunk_taps(a.hi, a.wi, a.pad, &plan->P.taps);
    if (!err.empty()) return err;
    if (!a.x || !a.y || !a.packed_w || !a.bias_pos || !a.bias || !a.err) return "trunk conv: null buffer";
    if (a.cap < 1 || a.cap > (int64_t)1 << 30) return "trunk conv: capacity out of range";
    if ((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.packed_w)) & 15) return "trunk conv: x and w must be 16-byte aligned";
    if ((reinterpret_cast<uintptr_t>(a.y) | reinterpret_cast<uintptr_t>(a.bias_pos) | reinterpret_cast<uintptr_t>(a.bias)) & 15) return "trunk conv: y and bias must be 16-byte aligned";
    EncodeTiledFn enc = encode_fn();
    if (!enc) return "trunk conv: cuTensorMapEncodeTiled is not available from this driver";
    const int n_in = a.hi * a.wi;
    {
        const cuuint64_t gdim[3] = {TRUNK_C, (cuuint64_t)n_in, (cuuint64_t)a.cap};
        const cuuint64_t gstride[2] = {TRUNK_C * 2, (cuuint64_t)n_in * TRUNK_C * 2};
        const cuuint32_t box[3] = {64, 1, TRUNK_BM};
        const cuuint32_t estr[3] = {1, 1, 1};
        CUresult rc = enc(&plan->amap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(a.x), gdim, gstride, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (rc != CUDA_SUCCESS) return "trunk conv: cuTensorMapEncodeTiled (x) failed (" + std::to_string((int)rc) + ")";
    }
    {
        const cuuint64_t gdim[2] = {TRUNK_C, 9 * TRUNK_C};
        const cuuint64_t gstride[1] = {TRUNK_C * 2};
        const cuuint32_t box[2] = {64, TRUNK_C};
        const cuuint32_t estr[2] = {1, 1};
        CUresult rc = enc(&plan->wmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(a.packed_w), gdim, gstride, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (rc != CUDA_SUCCESS) return "trunk conv: cuTensorMapEncodeTiled (w) failed (" + std::to_string((int)rc) + ")";
    }
    cudaError_t e = cudaFuncSetAttribute(k_trunk_conv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TK_SMEM);
    if (e != cudaSuccess) return std::string("trunk conv: shared memory opt-in: ") + cudaGetErrorString(e);
    plan->P.bias_pos = a.bias_pos;
    plan->P.bias = a.bias;
    plan->P.out = a.y;
    plan->P.err = a.err;
    plan->P.cap = a.cap;
    plan->n_sms = a.n_sms;
    plan->magic = TK_MAGIC;
    return "";
}

std::string trunk_launch(const TrunkPlan& plan, int64_t n, cudaStream_t st) {
    if (plan.magic != TK_MAGIC) return "trunk conv: not a plan (dbaz_nn_trunk_conv_plan)";
    if (n < 0 || n > plan.P.cap) return "trunk conv: n exceeds the capacity the plan was built for";
    if (n == 0) return "";
    TrunkParams P = plan.P;
    P.n = (int32_t)n;
    P.n_tiles = (int32_t)((n + TRUNK_BM - 1) / TRUNK_BM);
    P.n_items = P.n_tiles * P.taps.n_out;
    const int grid = P.n_items < plan.n_sms ? P.n_items : plan.n_sms;
    k_trunk_conv<<<grid, TK_THREADS, TK_SMEM, st>>>(plan.amap, plan.wmap, P);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? "" : std::string("k_trunk_conv: ") + cudaGetErrorString(e);
}

}  // namespace dbaz
