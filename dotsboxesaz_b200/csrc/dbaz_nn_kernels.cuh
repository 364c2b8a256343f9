// dbaz_nn_kernels.cuh -- fused stages of the leaf-evaluation pipeline.  The heads (log-softmax +
// exp, tanh) are one HBM pass here instead of PyTorch eager's several; the stem gathers the leaves
// and runs the first convolution with its bias / ReLU / eval-mode BatchNorm in one kernel.
//
// Reference semantics: dots_boxes/dots_boxes_nn.py:85-98 (x = bn(relu(conv(x)))), nn.py:49-58,
// nn.py:155-160 (p = exp(log_softmax), v = tanh).
#pragma once
#include <cuda/barrier>

#include "dbaz_device.cuh"

namespace dbaz {

template <typename T> struct Vec8;  // 8 consecutive channels
template <> struct Vec8<__nv_bfloat16> {
    uint4 raw;
    __device__ __forceinline__ void unpack(float* f) const {
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
        for (int i = 0; i < 4; ++i) { float2 t = __bfloat1622float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
    }
    __device__ __forceinline__ void pack(const float* f) {
        __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&raw);
#pragma unroll
        for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    }
};
template <> struct Vec8<__half> {
    uint4 raw;
    __device__ __forceinline__ void unpack(float* f) const {
        const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
        for (int i = 0; i < 4; ++i) { float2 t = __half22float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
    }
    __device__ __forceinline__ void pack(const float* f) {
        __half2* h = reinterpret_cast<__half2*>(&raw);
#pragma unroll
        for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
    }
};

// Heads: logits [n, ld] (policy logits in columns 0..A-1, value pre-activation in column A) ->
// priors float32 [n, A] = softmax (== exp(log_softmax), nn.py:159), values float32 [n] = tanh.
// One warp per row.
template <typename T>
__global__ void k_nn_heads(const T* __restrict__ logits, int ld, int A, float* __restrict__ priors,
                           float* __restrict__ values, int64_t n) {
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n) return;
    const T* row = logits + w * ld;
    float x[4];
    float m = -INFINITY;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int a = lane + 32 * k;
        x[k] = a < A ? (float)row[a] : -INFINITY;
        m = fmaxf(m, x[k]);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < 4; ++k) { x[k] = (lane + 32 * k < A) ? __expf(x[k] - m) : 0.0f; s += x[k]; }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    const float inv = 1.0f / s;
#pragma unroll
    for (int k = 0; k < 4; ++k) { int a = lane + 32 * k; if (a < A) priors[w * A + a] = x[k] * inv; }
    if (lane == 0) values[w] = tanhf((float)row[A]);
}

// The same with ResNetZero's value head finished in the kernel (nn.py:95-97): columns A .. A + n_hidden - 1 of the row are
// the value head's hidden pre-activations (fc0 output incl. bias); value = tanh(v_w[n_hidden] + sum_j relu(h_j) * v_w[j])
// (weights and bias of fc1 in one device vector, so that a weight reload needs no new kernel arguments).
// n_hidden <= 32.  One warp per row.
template <typename T>
__global__ void k_nn_heads_mlp(const T* __restrict__ logits, int ld, int A, int n_hidden, const float* __restrict__ v_w /* [n_hidden] weights, then the bias */,
                               float* __restrict__ priors, float* __restrict__ values, int64_t n) {
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n) return;
    const T* row = logits + w * ld;
    float x[4];
    float m = -INFINITY;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        int a = lane + 32 * k;
        x[k] = a < A ? (float)row[a] : -INFINITY;
        m = fmaxf(m, x[k]);
    }
    float hv = (lane < n_hidden) ? fmaxf((float)row[A + lane], 0.0f) * v_w[lane] : 0.0f;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
        hv += __shfl_xor_sync(0xffffffffu, hv, off);
    }
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < 4; ++k) { x[k] = (lane + 32 * k < A) ? __expf(x[k] - m) : 0.0f; s += x[k]; }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    const float inv = 1.0f / s;
#pragma unroll
    for (int k = 0; k < 4; ++k) { int a = lane + 32 * k; if (a < A) priors[w * A + a] = x[k] * inv; }
    if (lane == 0) values[w] = tanhf(hv + v_w[n_hidden]);
}

}  // namespace dbaz

namespace dbaz {

// ---------------------------------------------------------------------------------------------
// Stem: leaf gather + first 3x3 convolution + epilogue in ONE kernel, straight from the packed
// 32-byte leaf states (no plane tensor, no library call, no padding / cast / bias / ReLU / BN passes).
//
// The input planes of a leaf are two bit planes (edges) and one constant plane k = 2*boxes_to_close
// (dots_boxes_game.py:96-100), so with zero padding the convolution is, per output position p and
// channel co,
//     y[p][co] = B[p][co] + k * K2[p][co] + sum over (plane c in {0,1}, tap inside the board, edge bit set) W01[c][tap][co]
// where the host has folded into B / K2 / W01 (all float32, exact algebra): the conv bias, the optional
// input BatchNorm of ResNetZero (nn.py:118; its shift only contributes through in-board taps, hence the
// position dependence) and the third plane's weights summed over in-board taps.  The epilogue per output
// channel: mode 0 scale*relu(y)+shift (SimpleNN: conv -> ReLU -> BN), mode 1 relu(scale*y+shift) (ResNetZero:
// conv -> BN -> ReLU).
//
// Thread = (leaf, group of 8 output channels); all positions of a tile are accumulated in registers
// with the tap loop outermost, so each weight vector is read from shared memory once per leaf.  H, W
// are template parameters: every in-board test and bit index is a compile-time constant and padded
// taps cost nothing (31 % of a 4x4 map).  Output: [n][H][W][cout] (NHWC), 16-byte stores, a warp
// writes 512 contiguous bytes per position when cout == 256.
template <typename T, int H, int W, int MODE, int P0, int PN>
__device__ __noinline__ void stem_tile(const uint64_t e0, const uint64_t e1, const float kf, const float* __restrict__ w_s,
                                       const float* __restrict__ b_s, const float* __restrict__ k_s, const float* __restrict__ sc_s,
                                       const float* __restrict__ sh_s, T* __restrict__ out_leaf, int cout, int c0) {
    const int g = c0 >> 3, half4 = cout >> 3;  // swizzled shared layout, see k_nn_stem
    // the (up to 3 rows x W cols x 2 planes) input cells this tile touches, as 0.0f / 1.0f in registers;
    // indices are compile-time constants, unused entries are eliminated
    constexpr int R0 = (P0 / W) - 1, R1 = ((P0 + PN - 1) / W) + 1;  // row range touched (may fall outside the board)
    constexpr int NR = R1 - R0 + 1;
    float xv[2][NR][W];
#pragma unroll
    for (int c = 0; c < 2; ++c)
#pragma unroll
        for (int r = 0; r < NR; ++r)
#pragma unroll
            for (int x = 0; x < W; ++x) {
                const int hh = R0 + r;
                if (hh < 0 || hh >= H) { xv[c][r][x] = 0.0f; continue; }
                const int a = c * H * W + hh * W + x;
                const uint64_t bit = ((a < 64 ? e0 : e1) >> (a & 63)) & 1ull;
                xv[c][r][x] = __uint_as_float((unsigned)bit * 0x3f800000u);
            }
    float acc[PN][8];
#pragma unroll
    for (int p = 0; p < PN; ++p) {
        const float4* b4 = reinterpret_cast<const float4*>(b_s + (size_t)(P0 + p) * cout) + g;
        const float4* k4 = reinterpret_cast<const float4*>(k_s + (size_t)(P0 + p) * cout) + g;
        const float4 b0 = b4[0], b1 = b4[half4], k0 = k4[0], k1 = k4[half4];
        acc[p][0] = fmaf(kf, k0.x, b0.x); acc[p][1] = fmaf(kf, k0.y, b0.y); acc[p][2] = fmaf(kf, k0.z, b0.z); acc[p][3] = fmaf(kf, k0.w, b0.w);
        acc[p][4] = fmaf(kf, k1.x, b1.x); acc[p][5] = fmaf(kf, k1.y, b1.y); acc[p][6] = fmaf(kf, k1.z, b1.z); acc[p][7] = fmaf(kf, k1.w, b1.w);
    }
#pragma unroll
    for (int c = 0; c < 2; ++c)
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                asm volatile("" ::: "memory");  // keep one tap's weights live at a time
                const float4* wv = reinterpret_cast<const float4*>(w_s + (size_t)((c * 3 + ky) * 3 + kx) * cout) + g;
                const float4 w0 = wv[0], w1 = wv[half4];
#pragma unroll
                for (int p = 0; p < PN; ++p) {
                    const int h = (P0 + p) / W, x = (P0 + p) % W;
                    const int hh = h + ky - 1, ww = x + kx - 1;
                    if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;  // compile-time: padded taps cost nothing
                    const float xin = xv[c][hh - R0][ww];
                    acc[p][0] = fmaf(xin, w0.x, acc[p][0]); acc[p][1] = fmaf(xin, w0.y, acc[p][1]);
                    acc[p][2] = fmaf(xin, w0.z, acc[p][2]); acc[p][3] = fmaf(xin, w0.w, acc[p][3]);
                    acc[p][4] = fmaf(xin, w1.x, acc[p][4]); acc[p][5] = fmaf(xin, w1.y, acc[p][5]);
                    acc[p][6] = fmaf(xin, w1.z, acc[p][6]); acc[p][7] = fmaf(xin, w1.w, acc[p][7]);
                }
            }
    const float4* s4 = reinterpret_cast<const float4*>(sc_s) + g;
    const float4* t4 = reinterpret_cast<const float4*>(sh_s) + g;
    const float4 sa = s4[0], sb = s4[half4], ta = t4[0], tb = t4[half4];
    const float sc[8] = {sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z, sb.w}, sh[8] = {ta.x, ta.y, ta.z, ta.w, tb.x, tb.y, tb.z, tb.w};
#pragma unroll
    for (int p = 0; p < PN; ++p) {
        float y[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = (MODE == 0) ? fmaf(sc[j], fmaxf(acc[p][j], 0.0f), sh[j]) : fmaxf(fmaf(sc[j], acc[p][j], sh[j]), 0.0f);
        Vec8<T> v;
        v.pack(y);
        *reinterpret_cast<uint4*>(out_leaf + (size_t)(P0 + p) * cout + c0) = v.raw;
    }
}

// Persistent CTAs of 128 threads: the folded weights, both position tables and the epilogue parameters live in
// shared memory for the whole kernel; work is strided at leaf granularity (a group of cout/8 threads per leaf).
template <typename T, int H, int W, int MODE>
__global__ void __launch_bounds__(128, 4)
k_nn_stem(const dbaz_state* __restrict__ leaves, const float* __restrict__ w01 /*[18][cout]*/, const float* __restrict__ Bp /*[H*W][cout]*/,
          const float* __restrict__ K2 /*[H*W][cout]*/, const float* __restrict__ scale, const float* __restrict__ shift,
          T* __restrict__ out, int n, int cout) {
    extern __shared__ __align__(16) float smem_f[];
    constexpr int HW = H * W, TILE = (W <= 4 ? 2 * W : W);  // whole rows per tile
    float* w_s = smem_f;                 // [18][cout]
    float* b_s = w_s + 18 * cout;        // [HW][cout]
    float* k_s = b_s + HW * cout;        // [HW][cout]
    float* sc_s = k_s + HW * cout;       // [cout]
    float* sh_s = sc_s + cout;           // [cout]
    {   // table fill with 16-byte loads, 8 in flight per thread (scalar loads made this the whole kernel's cost).
        // Shared layout per row of `cout` floats: [half][group][4] -- a thread's channels 8g..8g+3 and 8g+4..8g+7 sit in
        // two planes so that each of its two LDS.128 is stride-16-bytes across the warp (conflict-free); the natural
        // layout puts lanes g and g+4 on the same banks.
        auto fill = [&](float* dst, const float* src, int count) {
            const float4* s4 = reinterpret_cast<const float4*>(src);
            float4* d4 = reinterpret_cast<float4*>(dst);
            const int n4 = count >> 2, row4 = cout >> 2, half4 = cout >> 3;
#pragma unroll 8
            for (int i = threadIdx.x; i < n4; i += blockDim.x) {
                const int row = i / row4, q = i - row * row4;  // q-th float4 of the row: channels 4q..4q+3
                d4[row * row4 + (q & 1) * half4 + (q >> 1)] = __ldg(s4 + i);
            }
        };
        fill(w_s, w01, 18 * cout);
        fill(b_s, Bp, HW * cout);
        fill(k_s, K2, HW * cout);
        fill(sc_s, scale, cout);
        fill(sh_s, shift, cout);
    }
    __syncthreads();
    const int groups = cout >> 3, per_block = blockDim.x / groups;
    const int g = threadIdx.x % groups, c0 = g << 3;
    for (int leaf = blockIdx.x * per_block + threadIdx.x / groups; leaf < n; leaf += gridDim.x * per_block) {
        const uint4 s0 = reinterpret_cast<const uint4*>(leaves + leaf)[0];
        const uint4 s1 = reinterpret_cast<const uint4*>(leaves + leaf)[1];
        const uint64_t e0 = (uint64_t)s0.x | ((uint64_t)s0.y << 32), e1 = (uint64_t)s0.z | ((uint64_t)s0.w << 32);
        const int to_play = s1.y & 0xffu;
        const int btc = to_play ? (int)(int16_t)(s1.x >> 16) : (int)(int16_t)(s1.x & 0xffffu);
        const float kf = (float)(int)(int8_t)btc;  // np.full_like(..., dtype=np.int8)
        T* o = out + (size_t)leaf * HW * cout;
#define DBAZ_STEM_TILE(I)                                                                                      \
        if constexpr (HW > (I) * TILE)                                                                           \
            stem_tile<T, H, W, MODE, (I) * TILE, (HW - (I) * TILE < TILE ? HW - (I) * TILE : TILE)>(e0, e1, kf, w_s, b_s, k_s, sc_s, sh_s, o, cout, c0);
        DBAZ_STEM_TILE(0) DBAZ_STEM_TILE(1) DBAZ_STEM_TILE(2) DBAZ_STEM_TILE(3) DBAZ_STEM_TILE(4) DBAZ_STEM_TILE(5)
#undef DBAZ_STEM_TILE
        static_assert(HW <= 6 * TILE, "position tiles");
    }
}


// ---------------------------------------------------------------------------------------------
// Stem on the tensor cores: the same leaf gather + first 3x3 convolution + ReLU as k_nn_stem, written as the small
// implicit GEMM it is,  D[row][co] = relu( sum_k A[row][k] * B[k][co] ),  row = leaf * H*W + position, K = 48:
//     k in [ 0, 18)  edge planes:   A = the edge bit under tap (plane k / 9, ky = k % 9 / 3, kx = k % 3), 0 outside the board
//     k in [18, 27)  third plane:   A = 2 * boxes_to_close[to_play] under an in-board tap (a small integer: exact in bf16 / fp16)
//     k in [27, 36)  in-board tap indicator (carries the shift of ResNetZero's input BatchNorm, nn.py:118)
//     k ==  36       1 (bias: conv bias and the folded output BatchNorm shift)
// B is folded on the host (nn.py: _stem_mma_table).  A is never materialised: a thread builds its m16n8k16 fragment
// from the two packed edge words of its two rows through a [position][k] code table in shared memory.  One warp
// owns a tile of 16 rows x (8 * NT) channels: 3 k-steps x NT `mma.sync` with fp32 accumulators, ReLU, then the tile goes
// through a padded shared-memory stage so that the global stores are 16 bytes per lane over contiguous rows.
// HBM-bound: 32 bytes in per leaf, H*W*cout*2 bytes out.
template <typename T> struct MmaType;
template <> struct MmaType<__nv_bfloat16> {
    static constexpr uint32_t ONE = 0x3F80u;
    static __device__ __forceinline__ uint32_t bits(float f) { return (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(f)); }
    static __device__ __forceinline__ void mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
        asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    }
    static __device__ __forceinline__ uint32_t pack_relu(float x, float y) {  // {relu(x), relu(y)} as bf16x2, one instruction
        uint32_t r;
        asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(y), "f"(x));
        return r;
    }
};
template <> struct MmaType<__half> {
    static constexpr uint32_t ONE = 0x3C00u;
    static __device__ __forceinline__ uint32_t bits(float f) { return (uint32_t)__half_as_ushort(__float2half_rn(f)); }
    static __device__ __forceinline__ void mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
        asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
    }
    static __device__ __forceinline__ uint32_t pack_relu(float x, float y) {
        uint32_t r;
        asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(y), "f"(x));
        return r;
    }
};

constexpr int STEM_K = 48;        // 3 k-steps of 16
constexpr int STEM_WARPS = 8;

// A-operand element for code c: 255 -> 0, < 128 -> edge bit c, 128 -> the third plane's value, 129 -> 1
template <typename T>
__device__ __forceinline__ uint32_t stem_a_elem(uint32_t c, const uint4& e, uint32_t kf_bits) {
    const uint32_t lo = (c & 64) ? e.z : e.x, hi = (c & 64) ? e.w : e.y;
    const uint32_t word = (c & 32) ? hi : lo;
    uint32_t v = ((word >> (c & 31)) & 1u) ? MmaType<T>::ONE : 0u;
    if (c & 128) v = (c == 128) ? kf_bits : (c == 129 ? MmaType<T>::ONE : 0u);
    return v;
}

// [48][cout] weights -> mma.sync B-fragment order [cout/8][3][32 lanes][4]: lane (g, t) of n-tile j, k-step s holds
// B[16s+2t][8j+g], B[16s+2t+1][8j+g], B[16s+2t+8][8j+g], B[16s+2t+9][8j+g]  (once per set of weights)
__global__ void k_nn_stem_mma_pack(const uint16_t* __restrict__ w48, uint2* __restrict__ packed, int cout) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (cout / 8) * 3 * 32) return;
    const int l = i & 31, js = i >> 5, s_ = js % 3, j = js / 3;
    const int gg = l >> 2, tt = l & 3, col = 8 * j + gg, k0 = 16 * s_ + 2 * tt;
    uint2 v;
    v.x = (uint32_t)w48[(size_t)k0 * cout + col] | ((uint32_t)w48[(size_t)(k0 + 1) * cout + col] << 16);
    v.y = (uint32_t)w48[(size_t)(k0 + 8) * cout + col] | ((uint32_t)w48[(size_t)(k0 + 9) * cout + col] << 16);
    packed[i] = v;
}

// nb != 0: write the output as planar tiles of the residual-tower kernel instead of NHWC
struct StemPlanar { int nb, wp, plane, buf; };

template <typename T, int NT>
__global__ void __launch_bounds__(STEM_WARPS * 32)
k_nn_stem_mma(const dbaz_state* __restrict__ leaves, const T* __restrict__ w48 /*fragment order, k_nn_stem_mma_pack*/, T* __restrict__ out,
              int n, int cout, int H, int W, StemPlanar pl) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NC = 8 * NT;                       // channels per work item
    constexpr int PARTS = NT >= 16 ? 2 : 1;          // the tile leaves through the stage in PARTS column parts
    constexpr int NTP = NT / PARTS, NCP = 8 * NTP;
    constexpr int STAGE_ROW = NCP * 2 + 16;          // bytes; +16 keeps the fragment stores conflict-free
    const int HW = H * W;
    const int n_chunks = cout / NC;
    uint2* b_s = reinterpret_cast<uint2*>(smem_raw);                                   // [cout/8][3][32] fragments, 8 bytes per lane
    unsigned char* code_s = smem_raw + (size_t)(cout / 8) * 3 * 32 * sizeof(uint2);    // [HW][48]
    unsigned char* stage_all = code_s + ((HW * STEM_K + 15) & ~15);                    // [STEM_WARPS][16][STAGE_ROW]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;

    // ---- B fragments, already in fragment order (k_nn_stem_mma_pack): ONE bulk asynchronous copy (TMA, cp.async.bulk)
    // global -> shared, issued by thread 0 and completed on an mbarrier while the other threads build the code table
    using block_barrier = cuda::barrier<cuda::thread_scope_block>;
    __shared__ block_barrier b_ready;
    if (threadIdx.x == 0) {
        init(&b_ready, blockDim.x);
        cuda::device::experimental::fence_proxy_async_shared_cta();
    }
    __syncthreads();
    block_barrier::arrival_token b_token;
    if (threadIdx.x == 0) {
        const unsigned b_bytes = (unsigned)((cout / 8) * 3 * 32 * sizeof(uint2));  // a multiple of 16; both ends 16-byte aligned
        cuda::device::memcpy_async_tx(reinterpret_cast<uint4*>(b_s), reinterpret_cast<const uint4*>(w48), cuda::aligned_size_t<16>(b_bytes), b_ready);
        b_token = cuda::device::barrier_arrive_tx(b_ready, 1, b_bytes);
    } else {
        b_token = b_ready.arrive();
    }
    // ---- code table
    for (int i = threadIdx.x; i < HW * STEM_K; i += blockDim.x) {
        const int pos = i / STEM_K, k = i - pos * STEM_K;
        const int y = pos / W, x = pos - y * W;
        unsigned char c = 255;
        if (k < 36) {
            const int tap = k % 9, yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
            if (yy >= 0 && yy < H && xx >= 0 && xx < W) c = (k < 18) ? (unsigned char)((k / 9) * HW + yy * W + xx) : (k < 27 ? 128 : 129);
        } else if (k == 36) c = 129;
        code_s[i] = c;
    }
    b_ready.wait(std::move(b_token));  // weights landed (and every thread has arrived)
    __syncthreads();

    unsigned char* stage = stage_all + (size_t)warp * 16 * STAGE_ROW;
    const uint32_t total_rows = (uint32_t)n * (uint32_t)HW;       // < 2^31, checked by the host
    const uint32_t n_tiles = (total_rows + 15u) >> 4;
    const uint32_t n_items = n_tiles * (uint32_t)n_chunks;
    for (uint32_t item = blockIdx.x * STEM_WARPS + warp; item < n_items; item += gridDim.x * STEM_WARPS) {
        const uint32_t tile = (n_chunks == 1) ? item : item / (uint32_t)n_chunks;
        const int chunk = (n_chunks == 1) ? 0 : (int)(item - tile * (uint32_t)n_chunks);
        const uint32_t r0 = tile << 4;
        // ---- A fragments of rows r0 + g and r0 + g + 8
        uint32_t a[3][4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t row = r0 + g + 8 * h;
            uint4 e = make_uint4(0, 0, 0, 0);
            uint32_t kfb = 0;
            uint32_t pos = 0;
            if (row < total_rows) {
                const uint32_t leaf = row / (uint32_t)HW;
                pos = row - leaf * (uint32_t)HW;
                e = reinterpret_cast<const uint4*>(leaves + leaf)[0];
                const uint2 s1 = reinterpret_cast<const uint2*>(leaves + leaf)[2];
                const int to_play = s1.y & 0xffu;
                const int btc = to_play ? (int)(int16_t)(s1.x >> 16) : (int)(int16_t)(s1.x & 0xffffu);
                kfb = MmaType<T>::bits((float)(int)(int8_t)btc);  // np.full_like(..., dtype=np.int8)
            }
            const unsigned char* cr = code_s + pos * STEM_K;
#pragma unroll
            for (int s_ = 0; s_ < 3; ++s_) {
                const uint32_t c01 = *reinterpret_cast<const uint16_t*>(cr + 16 * s_ + 2 * t);
                const uint32_t c89 = *reinterpret_cast<const uint16_t*>(cr + 16 * s_ + 2 * t + 8);
                a[s_][h] = stem_a_elem<T>(c01 & 0xffu, e, kfb) | (stem_a_elem<T>(c01 >> 8, e, kfb) << 16);
                a[s_][2 + h] = stem_a_elem<T>(c89 & 0xffu, e, kfb) | (stem_a_elem<T>(c89 >> 8, e, kfb) << 16);
            }
        }
        // ---- NT n-tiles x 3 k-steps in PARTS column parts: four independent accumulator chains in flight, ReLU, into
        // the stage, then 16 rows x NCP channels out with 16 bytes per lane (row segments contiguous)
        const uint2* bj = b_s + (size_t)chunk * NT * 3 * 32 + lane;
        unsigned char* st_lo = stage + (size_t)g * STAGE_ROW + 4 * t;
        unsigned char* st_hi = st_lo + 8 * STAGE_ROW;
        unsigned char* obase = reinterpret_cast<unsigned char*>(out) + ((size_t)r0 * cout + (size_t)chunk * NC) * 2;
        const uint32_t rows_here = min(16u, total_rows - r0);
#pragma unroll
        for (int part = 0; part < PARTS; ++part) {
            __syncwarp();
#pragma unroll
            for (int j0 = 0; j0 < NTP; j0 += 4) {
                float d[4][4];
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) { d[jj][0] = d[jj][1] = d[jj][2] = d[jj][3] = 0.0f; }
#pragma unroll
                for (int s_ = 0; s_ < 3; ++s_)
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const uint2 bb = bj[((part * NTP + j0 + jj) * 3 + s_) * 32];
                        MmaType<T>::mma(d[jj], a[s_], bb.x, bb.y);
                    }
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    *reinterpret_cast<uint32_t*>(st_lo + 16 * (j0 + jj)) = MmaType<T>::pack_relu(d[jj][0], d[jj][1]);
                    *reinterpret_cast<uint32_t*>(st_hi + 16 * (j0 + jj)) = MmaType<T>::pack_relu(d[jj][2], d[jj][3]);
                }
            }
            __syncwarp();
            constexpr int CH_PER_ROW = NCP * 2 / 16;  // 16-byte pieces per row segment
#pragma unroll 4
            if (pl.nb == 0) {
                for (int q = lane; q < 16 * CH_PER_ROW; q += 32) {
                    const int rr = q / CH_PER_ROW, cc = q % CH_PER_ROW;
                    if ((uint32_t)rr < rows_here) {
                        const uint4 v = *reinterpret_cast<const uint4*>(stage + (size_t)rr * STAGE_ROW + cc * 16);
                        *reinterpret_cast<uint4*>(obase + (size_t)rr * cout * 2 + (size_t)part * NCP * 2 + cc * 16) = v;
                    }
                }
            } else {
                // planar tiles of the residual-tower kernel (include/dbaz_b200.h: dbaz_nn_tower): consecutive rows of one
                // channel group are consecutive 16-byte slots, so lanes run over the rows
                for (int q = lane; q < 16 * CH_PER_ROW; q += 32) {
                    const int cc = q >> 4, rr = q & 15;
                    if ((uint32_t)rr < rows_here) {
                        const uint32_t row = r0 + (uint32_t)rr;
                        const uint32_t leaf = row / (uint32_t)HW, pos = row - leaf * (uint32_t)HW;
                        const uint32_t hh = pos / (uint32_t)W, ww = pos - hh * (uint32_t)W;
                        const uint32_t tile = leaf / (uint32_t)pl.nb, j = (leaf - tile * (uint32_t)pl.nb) * (uint32_t)pl.wp + ww;
                        const uint32_t cg = (uint32_t)(chunk * NC + part * NCP) / 8u + (uint32_t)cc;
                        const uint4 v = *reinterpret_cast<const uint4*>(stage + (size_t)rr * STAGE_ROW + cc * 16);
                        *reinterpret_cast<uint4*>(reinterpret_cast<unsigned char*>(out) + (size_t)tile * (size_t)pl.buf + 128 + (size_t)cg * (size_t)pl.plane +
                                                  (size_t)(hh * 128u + j) * 16) = v;
                    }
                }
            }
        }
    }
}

}  // namespace dbaz
