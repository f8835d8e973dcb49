// msw_conv.cuh -- the pieces of the tcgen05 3x3 convolutions (msw_conv_tc.cu, msw_cnn_fwd.cu) that must agree bit for
// bit between kernels: the nine-tap MMA issue, the fused GroupNorm statistics, the pooled-sum butterfly, the fp16
// stores and the P8 order of the fp32 residual stream.
//
// out[y][x][co] = sum_{dy,dx,ci} in[y+dy][x+dx][ci] * w[co][ci][dy][dx] is computed as nine shifted GEMMs per
// 128-pixel tile (8 image rows of one 16-wide board) that all accumulate into ONE TMEM accumulator.  The tile's input
// rows y0-1 .. y0+8 sit in shared memory as one linear [160 pixel][channel] block (K-major, swizzled), and a tap is
// nothing but a different shared-memory descriptor on that block:
//   * the A operand of tap (dy, dx) starts (dy+1) * 16 + dx pixels into the block.  The swizzle is a function of the
//     absolute shared-memory address (measured: descriptors whose start is shifted by whole 128- or 64-byte rows give
//     exact results with the matrix base offset left at 0), so no second copy and no im2col;
//   * a horizontal shift drags the neighbouring image row's edge pixel into the rows with x = 0 (dx = -1) or x = 15
//     (dx = +1); those rows of D are switched off for that tap with tcgen05.mma's disable-output-lane mask, which is
//     exactly the zero padding.  The first tap issued is the unmasked centre column, so every row of the accumulator
//     is initialised.
// K may be split into two channel blocks of different row widths (and swizzles), each with its own weight taps.
#pragma once

#include "msw_sm100.cuh"

#include <cuda_fp16.h>
#include <stdint.h>

namespace msw {

// The nine taps of one tile into accumulator `d`: KS0 16-channel k-steps of the first channel block (ROW0 bytes per
// pixel row, A block at a0, tap t's weights at w0 + t * w0_tap), then KS1 of the second (KS1 = 0: no second block).
// PAIR: the cta_group::2 form (M = 256, A rows 128 .. 255 are the peer CTA's tile), the mask covering both tiles.
// Called by one elected thread.
template <unsigned ROW0, int KS0, unsigned ROW1, int KS1, bool PAIR>
__device__ __forceinline__ void conv3x3_mmas(unsigned d, unsigned a0, unsigned a1, unsigned w0, unsigned w1,
                                             unsigned w0_tap, unsigned w1_tap, unsigned idesc)
{
    auto mma = [&](uint64_t a, uint64_t b, unsigned accumulate, unsigned mask) {
        if constexpr (PAIR) umma_f16_masked_pair(d, a, b, idesc, accumulate, mask);
        else umma_f16_masked(d, a, b, idesc, accumulate, mask);
    };
    unsigned accumulate = 0u;
#pragma unroll
    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
        for (int o = 0; o < 3; ++o) {
            const int dxi = o == 0 ? 1 : o == 1 ? 0 : 2;               // the unmasked centre tap first
            const int tap = dy * 3 + dxi;
            // rows of D whose horizontal neighbour is off the board: x = 0 for dx = -1, x = 15 for dx = +1
            const unsigned mask = dxi == 0 ? 0x00010001u : dxi == 2 ? 0x80008000u : 0u;
            const unsigned sa0 = a0 + (unsigned)((dy * 16 + dxi - 1) * (int)ROW0);
#pragma unroll
            for (int k = 0; k < KS0; ++k) {                            // 16 channels (32 bytes) per step
                mma(umma_desc<ROW0>(sa0) + 2u * k, umma_desc<ROW0>(w0 + tap * w0_tap) + 2u * k, accumulate, mask);
                accumulate = 1u;
            }
            if constexpr (KS1 > 0) {
                const unsigned sa1 = a1 + (unsigned)((dy * 16 + dxi - 1) * (int)ROW1);
#pragma unroll
                for (int k = 0; k < KS1; ++k)
                    mma(umma_desc<ROW1>(sa1) + 2u * k, umma_desc<ROW1>(w1 + tap * w1_tap) + 2u * k, 1u, mask);
            }
        }
}

// Deterministic warp sum: a fixed shuffle tree.
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Per-thread one-pass GroupNorm sums of v = x + bias over two 16-channel groups, shifted by a value of the warp's own
// data (no cancellation in S2 - S1^2 / n): group g has S1 = sum (v - shift[g]), S2 = sum (v - shift[g])^2.
struct GnSums {
    float shift[2], s1[2], s2[2];
};

// Adds this thread's 32 accumulator columns (lo, hi: channels 0..15, 16..31) to `s`.  h receives the conv output
// rounded to fp16 (the reference's rounding point) as 16 half2; the statistics are taken of those values plus cb2
// (the conv bias of the 32 channels).  `first`: the first call for these sums, which takes the shifts from lane 0.
__device__ __forceinline__ void gn_accumulate32(const uint32_t (&lo)[16], const uint32_t (&hi)[16], const float2 *cb2,
                                                bool first, uint32_t (&h)[16], GnSums &s)
{
#pragma unroll
    for (int jj = 0; jj < 16; ++jj) {
        const uint32_t *src = jj < 8 ? lo : hi;
        const __half2 hh = __floats2half2_rn(__uint_as_float(src[(2 * jj) & 15]), __uint_as_float(src[(2 * jj + 1) & 15]));
        h[jj] = *reinterpret_cast<const uint32_t *>(&hh);
        const float2 f = __half22float2(hh), cb = cb2[jj];
        const float v0 = f.x + cb.x, v1 = f.y + cb.y;
        const int g = jj >> 3;
        if (first && (jj & 7) == 0) s.shift[g] = __shfl_sync(0xffffffffu, v0, 0);
        const float d0 = v0 - s.shift[g], d1 = v1 - s.shift[g];
        s.s1[g] += d0 + d1;
        s.s2[g] = fmaf(d0, d0, fmaf(d1, d1, s.s2[g]));
    }
}

// (mean, M2) of COUNT values from their shifted sums S1, S2 (warp_sum of the per-thread sums).  Called by the one
// lane that stores the result: computed in every lane, it costs registers and reorders the epilogue.
template <int COUNT>
__device__ __forceinline__ float2 mean_m2(float shift, float s1, float s2)
{
    return make_float2(shift + s1 * (1.0f / COUNT), s2 - s1 * s1 * (1.0f / COUNT));
}

// One step of Chan et al.'s merge of (count na, mean, m2) with a partial of nb values: (mean_b, m2_b).  Exact
// division; callers merge their partials in a fixed order, so the result is bitwise reproducible.
__device__ __forceinline__ void chan_step(float &na, float &mean, float &m2, float nb, float mean_b, float m2_b)
{
    const float nn = na + nb, delta = mean_b - mean, w = nb / nn;
    mean = fmaf(delta, w, mean);
    m2 += m2_b + delta * delta * (na * w);
    na = nn;
}

// A channel's y = a*x + b from its group's (mean, M2) over COUNT values (biased variance, eps as torch), the affine
// gamma / beta, the conv bias `cb` (x is the conv output without it) and the Dropout2d scale `sc`: returns (a, b).
template <int COUNT>
__device__ __forceinline__ float2 gn_fold(float mean, float m2, float eps, float gamma, float beta, float cb, float sc)
{
    const float rg = rsqrtf(m2 * (1.0f / COUNT) + eps);
    const float a = gamma * rg;
    return make_float2(a * sc, fmaf(cb - mean, a, beta) * sc);
}

// Warp sum of 8 channels over the 32 lanes (pixels) in 9 shuffles, a fixed butterfly (deterministic): each step halves
// the number of channels a lane carries.  Returns the sum of channel `ch` = bit4*4 + bit3*2 + bit2 of the lane; lanes
// with (lane & 3) == 0 hold distinct channels.
__device__ __forceinline__ float pool8_butterfly(const float (&ps)[8], int lane, int &ch)
{
    const bool b4s = lane & 16, b3s = lane & 8, b2s = lane & 4;
    float a1[4], a2[2], a3;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        a1[i] = (b4s ? ps[4 + i] : ps[i]) + __shfl_xor_sync(0xffffffffu, b4s ? ps[i] : ps[4 + i], 16);
#pragma unroll
    for (int i = 0; i < 2; ++i)
        a2[i] = (b3s ? a1[2 + i] : a1[i]) + __shfl_xor_sync(0xffffffffu, b3s ? a1[i] : a1[2 + i], 8);
    a3 = (b2s ? a2[1] : a2[0]) + __shfl_xor_sync(0xffffffffu, b2s ? a2[0] : a2[1], 4);
    a3 += __shfl_xor_sync(0xffffffffu, a3, 2);
    a3 += __shfl_xor_sync(0xffffffffu, a3, 1);
    ch = (b4s ? 4 : 0) + (b3s ? 2 : 0) + (b2s ? 1 : 0);
    return a3;
}

__device__ __forceinline__ void st256(void *p, const uint32_t (&v)[8])
{
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void ld256(const void *p, uint32_t (&v)[8])
{
    asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "l"(p));
}

// 32 fp32 accumulator columns (lo, hi) -> fp16 at dst[0..31].  One 256-bit store per lane and 16 channels: the lanes of
// a warp write to 32 different 128-byte lines either way (pixels are C * 2 bytes apart), so the LSU cost is per
// instruction, not per byte.
__device__ __forceinline__ void store_half32(__half *dst, const uint32_t (&lo)[16], const uint32_t (&hi)[16])
{
#pragma unroll
    for (int c0 = 0; c0 < 32; c0 += 16) {
        const uint32_t *src = c0 == 0 ? lo : hi;
        uint32_t packed[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const __half2 hh = __floats2half2_rn(__uint_as_float(src[2 * k]), __uint_as_float(src[2 * k + 1]));
            packed[k] = *reinterpret_cast<const uint32_t *>(&hh);
        }
        st256(dst + c0, packed);
    }
}

// The fused epilogue's fp32 residual stream lives in HBM in the order the epilogue touches it -- "P8":
// [board][tile 2][channel slice SLICES][8-channel chunk 4][pixel 128][8 floats], a slice being the 32 channels of one
// epilogue warpgroup (SLICES = C / 32).  A thread (= pixel) owns one 32-byte chunk per (slice, chunk); the 32 lanes of a
// warp are 32 consecutive pixels, so every 256-bit load / store instruction of a warp covers 1 KB of consecutive
// addresses (8 full lines) instead of one line per lane as the pixel-major NHWC order would (32 lines per instruction:
// the epilogue was LSU-bound at 690 us per layer with it, against 240 us of MMAs).  Returns the float offset.
template <int SLICES>
__device__ __forceinline__ long long p8_offset(long long board, int tile, int slice, int c4, int pp)
{
    return ((((board * 2 + tile) * SLICES + slice) * 4 + c4) * 128 + pp) * 8;
}

}  // namespace msw
