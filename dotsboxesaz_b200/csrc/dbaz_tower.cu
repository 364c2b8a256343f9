// dbaz_tower.cu -- the residual tower of ResNetZero (reference nn.py:16-58: conv3x3 -> BN -> ReLU -> conv3x3 -> BN -> +x -> ReLU,
// 20 blocks of 64 channels in configuration.py:133-155) as ONE persistent sm_100a kernel: a tile of boards stays in
// shared memory through all 40 convolutions, the 3x3 weights stream from L2 by TMA, the products run on the 5th
// generation tensor cores (tcgen05.mma, accumulators in tensor memory) and the epilogue (folded BatchNorm bias,
// residual add, ReLU, bf16) writes the next layer's input straight back to shared memory.
//
// Why this shape.  Layer by layer (cuDNN) a 64-channel 3x3 convolution moves 256 bytes per position through HBM/L2 for
// 73.7 kFLOP -- at the ridge of the B200 roofline -- and a 128 x 64 x 16 MMA that fetches both operands from shared
// memory needs 192 B/clk of the SM's 128 B/clk.  Here
//   * activations never leave the SM: two buffers X, Y of [8 channel groups][H h-blocks][128 rows][8 channels] bf16;
//     a row is (board, w) with one zero pad column per board, so the tap (dy, dx) of output block h is simply block
//     h + dy read from a start address shifted by dx rows -- the unswizzled K-major operand layout with a row pitch
//     of 16 bytes makes any row a legal descriptor start, and the pad column supplies the zeros of the padding;
//   * the three dy taps of one dx share their A operand: ONE MMA of N = 192 multiplies input block h' with
//     [W(dy=+1) | W(dy=0) | W(dy=-1)] and accumulates into the accumulators of output blocks h'-1, h', h'+1, which are
//     neighbouring column ranges of tensor memory -- 107 B/clk of shared-memory operand traffic instead of 192, and
//     the taps that fall outside the board in y are never computed;
//   * weights: 12 chunks of 6 KB per convolution ((dx, 16 input channels) x 192 rows), a 5-slot ring filled by
//     cp.async.bulk.tensor (one elected thread) and released by tcgen05.commit;
//   * warp roles: 8 epilogue warps (tcgen05.ld -> bias/residual/ReLU -> st.shared), 1 weight producer, 1 MMA issuer,
//     1 tile loader; all hand-offs through mbarriers, no CTA-wide barrier inside the tile loop.
//
// Schedule of one stage (a 3x3 convolution): twelve passes p = 4 (dx + 1) + k over the weight chunks.  Passes 0..7
// stream chunk by chunk (h' inner); the last four (dx = +1) are consumed h'-outer, so that output block h is complete --
// tcgen05.commit on acc_full[h] -- as soon as input block h + 1 is through, and the epilogue drains it under the MMAs that
// remain.  The first pass of the NEXT stage waits block by block for the epilogue (act_ready[h]: block h written to the
// other buffer, its accumulator free) and splits its MMAs where an accumulator is touched for the first time
// (accumulate flag off).  Stage s odd reads the block input X as the residual and writes X in place; the optional last
// stage is the 1x1 head convolution (N = head_cout), whose epilogue -- like the last 3x3 stage's without a head -- goes to
// global memory.  Barriers: w_full / w_empty per weight slot, acc_full / act_ready per h-block, in_full per tile,
// tile_done per tile (a waiter is never more than one phase away from the barrier it polls; every wait is bounded).
// Measured on a B200 (DESIGN.md 4.1): 1397 TFLOP/s dense-equivalent at 15 984 boards of 5x5 (the sustained bf16 peak of
// the chip), tensor pipe 66 % of the cycles; the first version issued its MMAs from divergent single-thread code and
// reached 445 -- a dozen dependent scalar instructions per MMA cost more than the MMA.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <string>

#include "dbaz_tcgen05.cuh"
#include "dbaz_tower.cuh"

namespace dbaz {

namespace {

constexpr int EPI_WARPS = 8;
constexpr int W_WARP = EPI_WARPS;        // weight producer
constexpr int MMA_WARP = EPI_WARPS + 1;  // MMA issuer, owns the tensor-memory allocation
constexpr int IO_WARP = EPI_WARPS + 2;   // tile loader
constexpr int THREADS = (EPI_WARPS + 3) * 32;
constexpr int NSLOT = 5;
constexpr int MAXH = 6;
constexpr uint32_t TMEM_COLS = 512;

struct TowerParams {
    const unsigned char* blob;
    const unsigned char* packed_w;
    const float* bias;
    __nv_bfloat16* out;
    int n_stages, head_cout;
    int n_boards, n_tiles;
    int H, W, WP, nb, plane, buf;
    int* err;
    long long* dbg;  // optional timeline of CTA 0's first tile (clock64): [stage][16]
};

// ---------------------------------------------------------------- the kernel
template <int H>
__global__ void __launch_bounds__(THREADS, 1)
k_resnet_tower(const __grid_constant__ CUtensorMap wmap, const TowerParams P) {
    extern __shared__ unsigned char smem_dyn[];
    const uint32_t raw = smem_u32(smem_dyn);
    const uint32_t base = (raw + 127u) & ~127u;
    unsigned char* const gbase = smem_dyn + (base - raw);
    const int PLANE = P.plane, BUF = P.buf;
    const uint32_t X = base, Y = base + (uint32_t)BUF, WS = base + 2u * (uint32_t)BUF;
    const uint32_t BAR = WS + NSLOT * TOWER_CHUNK_BYTES;
    // barriers (8 bytes each)
    const uint32_t w_full = BAR, w_empty = BAR + 8 * NSLOT, acc_full = BAR + 16 * NSLOT, act_ready = acc_full + 8 * MAXH,
                   in_full = act_ready + 8 * MAXH, tile_done = in_full + 8, tmem_slot = tile_done + 8;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;  // provably warp-uniform
    const int S3 = P.n_stages, S = S3 + (P.head_cout ? 1 : 0);

    // ---- one-time setup: zero both activation buffers (pads and guard rows must read as zero), barriers, tensor memory
    {
        uint4* z = reinterpret_cast<uint4*>(gbase);
        const int n16 = (2 * BUF) >> 4;
        for (int i = threadIdx.x; i < n16; i += THREADS) z[i] = make_uint4(0, 0, 0, 0);
    }
    if (threadIdx.x == 0) {
        for (int i = 0; i < NSLOT; ++i) { mbar_init(w_full + 8 * i, 1); mbar_init(w_empty + 8 * i, 1); }
        for (int i = 0; i < MAXH; ++i) { mbar_init(acc_full + 8 * i, 1); mbar_init(act_ready + 8 * i, EPI_WARPS * 32); }
        mbar_init(in_full, 1);
        mbar_init(tile_done, EPI_WARPS * 32);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(tmem_slot));

    const int my_tiles = (P.n_tiles > (int)blockIdx.x) ? (P.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    if (warp == W_WARP) {
        // =================== weight producer: one thread streams the chunks of every stage of every tile
        if (lane == 0) {
            uint32_t n = 0;
            for (int it = 0; it < my_tiles; ++it) {
                for (int s = 0; s < S; ++s) {
                    const int chunks = (s < S3) ? TOWER_CHUNKS_PER_STAGE : 1;
                    for (int p = 0; p < chunks; ++p, ++n) {
                        const uint32_t slot = n % NSLOT, round = n / NSLOT;
                        mbar_wait(w_empty + 8 * slot, (round & 1u) ^ 1u, P.err, 1);
                        const uint32_t dst = WS + slot * TOWER_CHUNK_BYTES;
                        if (s < S3) {
                            mbar_expect_tx(w_full + 8 * slot, TOWER_CHUNK_BYTES);
                            tma_load_2d(dst, &wmap, 0, (s * TOWER_CHUNKS_PER_STAGE + p) * 48, w_full + 8 * slot);
                        } else {
                            const uint32_t bytes = (uint32_t)P.head_cout * 128u;
                            mbar_expect_tx(w_full + 8 * slot, bytes);
                            bulk_load(dst, P.packed_w + (size_t)S3 * TOWER_CHUNKS_PER_STAGE * TOWER_CHUNK_BYTES, bytes, w_full + 8 * slot);
                        }
                    }
                }
            }
        }
    } else if (warp == IO_WARP) {
        // =================== tile loader: the planar tile image goes to X as eight bulk copies
        if (lane == 0) {
            for (int it = 0; it < my_tiles; ++it) {
                const int tile = (int)blockIdx.x + it * (int)gridDim.x;
                // X is free once the last stage of the previous tile is through its epilogue (which read X as the residual,
                // after the MMAs that read X).  A barrier of its own, one phase per tile: a waiter may never be two
                // phases away from the barrier it polls, and act_ready runs through S phases per tile.
                if (it > 0) mbar_wait(tile_done, (uint32_t)(it - 1) & 1u, P.err, 2);
                mbar_expect_tx(in_full, 8u * (uint32_t)PLANE);
                const unsigned char* src = P.blob + (size_t)tile * (size_t)BUF + 128;
                for (int cg = 0; cg < 8; ++cg) bulk_load(X + 128 + cg * PLANE, src + (size_t)cg * PLANE, (uint32_t)PLANE, in_full);
            }
        }
    } else if (warp == MMA_WARP) {
        // =================== MMA issuer.  The whole warp runs the control flow (warp-uniform, so descriptors stay in
        // uniform registers and the h' loops unroll with immediate offsets); one elected lane issues the MMAs and commits.
        // A single thread pays its own instruction latency for every operation: a dozen dependent instructions per MMA
        // already cost more than the 96 clocks the tensor core needs for it.
        uint32_t n = 0, g = 0;
        const uint32_t a_lbo = ((uint32_t)PLANE >> 4) << 16, b_lbo = (3072u >> 4) << 16;
        for (int it = 0; it < my_tiles; ++it) {
            mbar_wait(in_full, it & 1, P.err, 3);
            for (int s = 0; s < S; ++s, ++g) {
                const uint32_t src = (s & 1) ? Y : X;  // the head stage (s == S3, S3 even) reads X
                const uint32_t prev_par = (g - 1u) & 1u;
                const bool trace = P.dbg && blockIdx.x == 0 && it == 0 && s < 64;
                if (s < S3) {
                    if (trace && lane == 0) P.dbg[s * 16 + 0] = clock64();
                    // ---- passes 0..7 (dx = -1, 0; four K steps each): one weight chunk per pass, h' inner
                    for (int p = 0; p < 8; ++p, ++n) {
                        const uint32_t slot = n % NSLOT, round = n / NSLOT;
                        mbar_wait(w_full + 8 * slot, round & 1u, P.err, 4);
                        tc_fence_after();
                        const int dx = (p >> 2) - 1, k = p & 3;
                        const uint32_t a_lo = (((src + 128u + (uint32_t)(2 * k) * (uint32_t)PLANE + (uint32_t)(dx * 16)) >> 4) & 0x3fffu) | a_lbo;
                        const uint32_t b_lo = (((WS + slot * TOWER_CHUNK_BYTES) >> 4) & 0x3fffu) | b_lbo;
                        if (p == 0) {
                            // first pass of a stage: input block hp must be written and accumulators hp-1..hp+1 drained by the
                            // previous stage's epilogue; blocks hp-1, hp already hold a partial sum, block hp+1 is touched first
#pragma unroll
                            for (int hp = 0; hp < H; ++hp) {
                                if (hp == 0) mbar_wait(act_ready, prev_par, P.err, 5);
                                if (hp + 1 < H) mbar_wait(act_ready + 8 * (hp + 1), prev_par, P.err, 5);
                                tc_fence_after();
                                if (elect_one()) {
                                    const uint64_t ad = desc64(a_lo + (uint32_t)hp * 128u);
                                    if (hp == 0) {
                                        umma(tmem, ad, desc64(b_lo + 64u), umma_idesc(128), 0u);
                                    } else {
                                        umma(tmem + 64u * (hp - 1), ad, desc64(b_lo), umma_idesc(128), 1u);
                                        if (hp + 1 < H) umma(tmem + 64u * (hp + 1), ad, desc64(b_lo + 128u), umma_idesc(64), 0u);
                                    }
                                }
                                __syncwarp();
                            }
                        } else if (elect_one()) {
#pragma unroll
                            for (int hp = 0; hp < H; ++hp) {
                                const int lo = hp > 0 ? hp - 1 : 0, hi = hp + 1 < H ? hp + 1 : H - 1;
                                umma(tmem + 64u * lo, desc64(a_lo + (uint32_t)hp * 128u), desc64(b_lo + (uint32_t)(lo - (hp - 1)) * 64u),
                                     umma_idesc(64u * (hi - lo + 1)), 1u);
                            }
                        }
                        __syncwarp();
                        if (elect_one()) umma_commit(w_empty + 8 * slot);
                        __syncwarp();
                        if (trace && lane == 0 && p <= 1) P.dbg[s * 16 + 1 + p] = clock64();
                    }
                    // ---- passes 8..11 (dx = +1): all four chunks, then h' OUTER, so that output block h is complete as soon as
                    // input block h + 1 is through and the epilogue drains it under the remaining MMAs
                    uint32_t b_lo4[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t slot = (n + k) % NSLOT, round = (n + k) / NSLOT;
                        mbar_wait(w_full + 8 * slot, round & 1u, P.err, 4);
                        b_lo4[k] = (((WS + slot * TOWER_CHUNK_BYTES) >> 4) & 0x3fffu) | b_lbo;
                    }
                    tc_fence_after();
                    const uint32_t a_lo = (((src + 128u + 16u) >> 4) & 0x3fffu) | a_lbo;
                    const uint32_t a_kstep = (2u * (uint32_t)PLANE) >> 4;
                    if (elect_one()) {
#pragma unroll
                        for (int hp = 0; hp < H; ++hp) {
                            const int lo = hp > 0 ? hp - 1 : 0, hi = hp + 1 < H ? hp + 1 : H - 1;
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                umma(tmem + 64u * lo, desc64(a_lo + (uint32_t)k * a_kstep + (uint32_t)hp * 128u),
                                     desc64(b_lo4[k] + (uint32_t)(lo - (hp - 1)) * 64u), umma_idesc(64u * (hi - lo + 1)), 1u);
                            if (hp >= 1) umma_commit(acc_full + 8 * (hp - 1));
                            if (hp == H - 1) umma_commit(acc_full + 8 * hp);
                        }
#pragma unroll
                        for (int k = 0; k < 4; ++k) umma_commit(w_empty + 8 * ((n + k) % NSLOT));
                    }
                    __syncwarp();
                    n += 4;
                    if (trace && lane == 0) P.dbg[s * 16 + 3] = clock64();
                } else {
                    // fused 1x1 head convolution: N = head_cout, four K steps, one weight chunk
                    const uint32_t slot = n % NSLOT, round = n / NSLOT;
                    mbar_wait(w_full + 8 * slot, round & 1u, P.err, 4);
                    tc_fence_after();
                    const uint32_t hc = (uint32_t)P.head_cout;
                    const uint32_t a_lo = (((src + 128u) >> 4) & 0x3fffu) | a_lbo;
                    const uint32_t a_kstep = (2u * (uint32_t)PLANE) >> 4;
                    const uint32_t b_lo = (((WS + slot * TOWER_CHUNK_BYTES) >> 4) & 0x3fffu) | (((hc * 16u) >> 4) << 16);
                    const uint32_t idesc = umma_idesc(hc);
#pragma unroll
                    for (int hp = 0; hp < H; ++hp) {
                        mbar_wait(act_ready + 8 * hp, prev_par, P.err, 5);
                        tc_fence_after();
                        if (elect_one()) {
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                umma(tmem + 64u * hp, desc64(a_lo + (uint32_t)k * a_kstep + (uint32_t)hp * 128u), desc64(b_lo + (uint32_t)k * hc * 2u), idesc,
                                     k > 0 ? 1u : 0u);
                            umma_commit(acc_full + 8 * hp);
                        }
                        __syncwarp();
                    }
                    if (elect_one()) umma_commit(w_empty + 8 * slot);
                    __syncwarp();
                    ++n;
                }
            }
        }
    } else {
        // =================== epilogue warps: warp w drains lanes 32 (w % 4) .. +31, columns 32 (w / 4) .. +31 of a block
        const int q = warp & 3, half = warp >> 2;
        const int row = 32 * q + lane;                 // row inside an h-block = accumulator lane
        const int bi = row / P.WP, w = row - bi * P.WP;
        const bool row_ok = bi < P.nb && w < P.W;
        uint32_t g = 0;
        for (int it = 0; it < my_tiles; ++it) {
            const int tile = (int)blockIdx.x + it * (int)gridDim.x;
            const int board = tile * P.nb + bi;
            const bool store_ok = row_ok && board < P.n_boards;
            for (int s = 0; s < S; ++s, ++g) {
                const bool head = s >= S3, last = s == S - 1;
                const bool residual = !head && (s & 1);
                const uint32_t dst = (s & 1) ? X : Y;
                const bool active = !head || half == 0;  // the head has at most 32 columns: the upper half has nothing to drain
                float b[32];
                if (active) {
                    const float4* bp = reinterpret_cast<const float4*>(P.bias + (size_t)s * TOWER_C + 32 * half);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 v = __ldg(bp + i);
                        b[4 * i] = v.x; b[4 * i + 1] = v.y; b[4 * i + 2] = v.z; b[4 * i + 3] = v.w;
                    }
                }
                const bool trace = P.dbg && blockIdx.x == 0 && it == 0 && s < 64 && threadIdx.x == 0;
                for (int h = 0; h < H; ++h) {
                    mbar_wait(acc_full + 8 * h, g & 1u, P.err, 6);
                    tc_fence_after();
                    if (trace) P.dbg[s * 16 + 4 + 2 * h] = clock64();
                    if (active) {
                        uint32_t r[32];
                        tmem_ld32(tmem + ((uint32_t)(32 * q) << 16) + 64u * h + 32u * half, r);
                        const uint32_t cell = (uint32_t)(h * 128 + row) * 16u + 128u + (uint32_t)(4 * half) * (uint32_t)PLANE;
                        uint4 res[4] = {};
                        if (residual) {
#pragma unroll
                            for (int c = 0; c < 4; ++c)
                                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                                             : "=r"(res[c].x), "=r"(res[c].y), "=r"(res[c].z), "=r"(res[c].w)
                                             : "r"(dst + cell + (uint32_t)c * (uint32_t)PLANE));
                        }
                        tmem_ld_wait();
                        // bias (+ residual) in fp32, ReLU inside the conversion to bf16x2; rows that hold no board point
                        // (pad column, guard rows) are written as zeros: they are the zero padding of the next convolution
                        uint32_t o[16];
                        if (row_ok) {
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const uint32_t rr[4] = {res[c].x, res[c].y, res[c].z, res[c].w};
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    const int i = 8 * c + 2 * e;
                                    float v0 = __uint_as_float(r[i]) + b[i], v1 = __uint_as_float(r[i + 1]) + b[i + 1];
                                    if (residual) { v0 += bf16_lo(rr[e]); v1 += bf16_hi(rr[e]); }
                                    o[4 * c + e] = pack_relu_bf16(v0, v1);
                                }
                            }
                        } else {
#pragma unroll
                            for (int i = 0; i < 16; ++i) o[i] = 0u;
                        }
                        if (!last) {
#pragma unroll
                            for (int c = 0; c < 4; ++c)
                                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(dst + cell + (uint32_t)c * (uint32_t)PLANE),
                                             "r"(o[4 * c]), "r"(o[4 * c + 1]), "r"(o[4 * c + 2]), "r"(o[4 * c + 3])
                                             : "memory");
                        } else if (store_ok) {
                            const int cout = head ? P.head_cout : TOWER_C;
                            uint4* op = reinterpret_cast<uint4*>(P.out + ((size_t)((size_t)board * H + h) * P.W + w) * cout + 32 * half);
                            const int n16 = head ? (cout >> 3) : 4;
#pragma unroll
                            for (int c = 0; c < 4; ++c)
                                if (c < n16) op[c] = make_uint4(o[4 * c], o[4 * c + 1], o[4 * c + 2], o[4 * c + 3]);
                        }
                    }
                    fence_proxy_async();   // the next stage's MMAs read what was just stored through the async proxy
                    tc_fence_before();
                    mbar_arrive(act_ready + 8 * h);
                    if (trace) P.dbg[s * 16 + 5 + 2 * h] = clock64();
                }
            }
            mbar_arrive(tile_done);
        }
    }
    // ---- teardown
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
    }
}

// NHWC [n][H][W][64] bf16 -> planar tiles.  One thread per 16-byte piece (position, channel group).
__global__ void k_tower_planarize(const uint4* __restrict__ nhwc, unsigned char* __restrict__ blob, int64_t n_pieces, int H, int W, int WP,
                                  int nb, int plane, int buf) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pieces) return;
    const int cg = (int)(i & 7);
    const int64_t pos = i >> 3;
    const int w = (int)(pos % W);
    const int64_t t = pos / W;
    const int h = (int)(t % H);
    const int64_t board = t / H;
    const int64_t tile = board / nb;
    const int j = (int)(board - tile * nb) * WP + w;
    *reinterpret_cast<uint4*>(blob + tile * (int64_t)buf + 128 + (int64_t)cg * plane + (int64_t)(h * 128 + j) * 16) = nhwc[i];
}

}  // namespace

TowerGeom tower_geom(int H, int W) {
    TowerGeom g;
    g.H = H; g.W = W; g.WP = W + 1;
    g.nb = 128 / g.WP;
    g.plane = H * 128 * 16 + 128;
    g.buf = 128 + 8 * g.plane;
    g.ok = (H >= 2 && H <= MAXH && g.WP <= 128 && W >= 1) ? 1 : 0;
    return g;
}

std::string tower_planarize(const TowerGeom& g, const void* nhwc, void* blob, int64_t n, cudaStream_t st) {
    if (!g.ok) return "tower: unsupported board";
    const int64_t pieces = n * g.H * g.W * 8;
    if (pieces == 0) return "";
    k_tower_planarize<<<(unsigned)((pieces + 255) / 256), 256, 0, st>>>(reinterpret_cast<const uint4*>(nhwc), reinterpret_cast<unsigned char*>(blob),
                                                                        pieces, g.H, g.W, g.WP, g.nb, g.plane, g.buf);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? "" : std::string("k_tower_planarize: ") + cudaGetErrorString(e);
}

std::string tower_launch(const TowerGeom& g, const TowerLaunch& a, cudaStream_t st) {
    if (!g.ok) return "tower: unsupported board (2 <= L+1 <= 6)";
    if (a.n_stages < 1) return "tower: n_stages must be >= 1";
    if (a.head_cout != 0 && (a.head_cout % 16 != 0 || a.head_cout > 32 || (a.n_stages & 1))) return "tower: head_cout must be 16 or 32 after an even number of stages";
    if (a.n_boards <= 0) return "";
    EncodeTiledFn enc = encode_fn();
    if (!enc) return "tower: cuTensorMapEncodeTiled is not available from this driver";
    CUtensorMap wmap;
    const cuuint64_t rows = (cuuint64_t)a.n_stages * TOWER_CHUNKS_PER_STAGE * 48;
    const cuuint64_t gdim[2] = {64, rows};
    const cuuint64_t gstride[1] = {128};
    const cuuint32_t box[2] = {64, 48};
    const cuuint32_t estr[2] = {1, 1};
    CUresult rc = enc(&wmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(a.packed_w), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) return "tower: cuTensorMapEncodeTiled failed (" + std::to_string((int)rc) + ")";
    TowerParams P;
    P.blob = reinterpret_cast<const unsigned char*>(a.blob);
    P.packed_w = reinterpret_cast<const unsigned char*>(a.packed_w);
    P.bias = a.bias;
    P.out = reinterpret_cast<__nv_bfloat16*>(a.out);
    P.n_stages = a.n_stages; P.head_cout = a.head_cout;
    P.n_boards = (int)a.n_boards;
    P.n_tiles = (int)((a.n_boards + g.nb - 1) / g.nb);
    P.H = g.H; P.W = g.W; P.WP = g.WP; P.nb = g.nb; P.plane = g.plane; P.buf = g.buf;
    P.err = a.err_flag;
    P.dbg = a.dbg;
    // the shared-memory size depends on H only (g.buf), so one opt-in per instantiation is enough
    const size_t smem = 128 + 2 * (size_t)g.buf + NSLOT * TOWER_CHUNK_BYTES + 8 * (2 * NSLOT + 2 * MAXH + 2) + 16;
    const int grid = P.n_tiles < a.n_sms ? P.n_tiles : a.n_sms;
    cudaError_t e = cudaSuccess;
#define DBAZ_TOWER_H(HH)                                                                                       \
    case HH: {                                                                                                 \
        static bool opted = false;                                                                             \
        if (!opted) {                                                                                          \
            e = cudaFuncSetAttribute(k_resnet_tower<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
            if (e != cudaSuccess) return std::string("tower: shared memory opt-in: ") + cudaGetErrorString(e); \
            opted = true;                                                                                      \
        }                                                                                                      \
        k_resnet_tower<HH><<<grid, THREADS, smem, st>>>(wmap, P);                                              \
        break;                                                                                                 \
    }
    switch (g.H) {
        DBAZ_TOWER_H(2) DBAZ_TOWER_H(3) DBAZ_TOWER_H(4) DBAZ_TOWER_H(5) DBAZ_TOWER_H(6)
        default: return "tower: unsupported board";
    }
#undef DBAZ_TOWER_H
    e = cudaGetLastError();
    return e == cudaSuccess ? "" : std::string("k_resnet_tower: ") + cudaGetErrorString(e);
}

}  // namespace dbaz
