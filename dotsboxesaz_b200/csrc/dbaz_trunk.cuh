// dbaz_trunk.cuh -- host-side interface of the trunk convolution kernel (dbaz_trunk.cu), shared with dbaz_capi.cu.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>

namespace dbaz {

constexpr int TRUNK_C = 256;        // input and output channels (SimpleNN: N_CH)
constexpr int TRUNK_MAX_POS = 64;   // points of the largest board the engine plays (2 (L+1)(C+1) <= 128 actions)
constexpr int TRUNK_BM = 128;       // boards per work item (the M of one tcgen05.mma)

// Taps of every output position of a 3x3 convolution (stride 1, zero padding `pad`) over an hi x wi grid: position
// p = y * wo + x takes count[p] taps; tap k is (tap[p][k] & 15) = 3 ky + kx of the weights applied to input position
// (tap[p][k] >> 4), k ascending in (ky, kx) -- the order of the taps inside each 64-channel chunk of the K loop.  Taps that fall into the padding are left out.  order[] lists the output
// positions by descending tap count (ties by position), the order in which the work items are handed out.
struct TrunkTaps {
    int32_t hi, wi, pad, ho, wo, n_out;
    uint8_t count[TRUNK_MAX_POS];
    uint8_t order[TRUNK_MAX_POS];
    uint16_t tap[TRUNK_MAX_POS][9];
};
std::string trunk_taps(int hi, int wi, int pad, TrunkTaps* t);

struct TrunkParams {
    TrunkTaps taps;
    const float* bias_pos;   // [n_out][256] float32
    const float* bias;       // [256] float32
    void* out;               // [cap][n_out][256] bf16
    int* err;                // device int: set non-zero if a barrier wait timed out
    int64_t cap;             // boards the buffers hold
    int32_t n, n_tiles, n_items, reserved;
};

// Everything one layer's launches need, built once per (buffers, weights) by trunk_plan: the tensor maps are encoded
// over the buffers' full capacity, so launching for any n <= cap allocates, encodes and configures nothing.
struct alignas(64) TrunkPlan {
    CUtensorMap amap;        // x [cap][hi * wi][256] bf16, box {64 channels, 1 position, 128 boards}, 128-byte swizzle
    CUtensorMap wmap;        // w [9 * 256][256] bf16, box {64 input channels, 256 output channels}, 128-byte swizzle
    TrunkParams P;
    int32_t n_sms, magic;
};

struct TrunkPlanArgs {
    const void* x;           // [cap][hi][wi][256] bf16 (NHWC)
    void* y;                 // [cap][ho][wo][256] bf16 (NHWC)
    const void* packed_w;    // [ky][kx][cout][cin] bf16
    const float* bias_pos;   // [ho * wo][256] float32
    const float* bias;       // [256] float32
    int64_t cap;
    int hi, wi, pad, n_sms;
    int* err;
};
std::string trunk_plan(const TrunkPlanArgs& a, TrunkPlan* plan);
std::string trunk_launch(const TrunkPlan& plan, int64_t n, cudaStream_t st);

}  // namespace dbaz
