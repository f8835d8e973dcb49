// msw_conv_tc.cu -- 3x3 "same" convolution of the policy trunk (96 -> 96 channels on 16x16 boards, and the stem's
// 16 -> 96; fp16 NHWC in, fp32 accumulate, fp16 NHWC out) on the 5th-generation tensor cores, plain
// (conv3x3_tc_kernel<false>: no bias, it is folded into msw_gn_act) or with GroupNorm / ReLU / Dropout2d /
// residual add (and the value head's average pool) fused into the epilogue (conv3x3_tc_kernel<true>).
// 128 -> 128 channels (and the stem's 16 -> 128) run on conv3x3_pair_kernel below: one board per CTA pair.
//
// out[y][x][co] = sum_{dy,dx,ci} in[y+dy][x+dx][ci] * w[co][ci][dy][dx] is computed as nine shifted GEMMs
// per 128-pixel tile (8 image rows of one board) that all accumulate into ONE TMEM accumulator.  The tile's
// input rows y0-1 .. y0+8 sit in shared memory as one linear [160 pixel][96 ch] block (a single 4-D TMA box;
// rows above / below the board are zero-filled by the tensor map), and a tap is nothing but a different
// shared-memory descriptor on that block:
//   * the A operand of tap (dy, dx) starts (dy+1) * 16 + dx pixels into the block.  The swizzle is a function
//     of the absolute shared-memory address (measured: descriptors whose start is shifted by whole 128- or
//     64-byte rows give exact results with the matrix base offset left at 0), so no second copy and no im2col;
//   * a horizontal shift drags the neighbouring image row's edge pixel into the rows with x = 0 (dx = -1) or
//     x = 15 (dx = +1); those rows of D are switched off for that tap with tcgen05.mma's disable-output-lane
//     mask, which is exactly the zero padding.  The first tap issued is the unmasked centre column, so every
//     row of the accumulator is initialised.
// All nine [96 x 96] weight taps stay resident in shared memory (162 KB, loaded once per persistent CTA);
// the activation streams through a 2-stage ring.  K = 96 = one 64-channel block (128-byte swizzle) + one
// 32-channel block (64-byte swizzle).  Roles: warp 0 TMA producer, warp 1 MMA issuer (54 tcgen05.mma of
// 128 x 96 x 16 per tile into a ring of four 96-column accumulators), warp 2 TMEM allocation, warps 4-15
// epilogue (thread = pixel, each warpgroup a third of the channels).  The mbarrier / TMA / tcgen05 wrappers are in
// msw_sm100.cuh.
#include "../../include/msw_b200.h"
#include "msw_common.cuh"
#include "msw_error.h"
#include "msw_sm100.cuh"

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

// Ablation switches for tools/convgn_ablation.py: compiled in only with -DMSW_DEV_KNOBS (the product library has none).
#ifdef MSW_DEV_KNOBS
#define MSW_DBG(bit) ((dbg & (bit)) != 0)
#else
#define MSW_DBG(bit) false
#endif

namespace msw {

namespace cv {
constexpr int C = 96, HW_W = 16, TILE_PX = 128, ROWS_IN = 10, PX_IN = ROWS_IN * HW_W;   // C = output channels; 160 staged pixels
constexpr int THREADS = 512, STAGES = 2, TMEM_COLS = 512;       // 4 control warps + 12 epilogue warps
constexpr int ACC = 4;                                                   // accumulator ring: 4 x 96 TMEM columns

// Shared-memory plan for CIN input channels.  CIN = 96: K = one 64-channel block (128-byte rows, 128-byte
// swizzle) + one 32-channel block (64-byte rows, 64-byte swizzle).  CIN = 16 (the stem, observation planes padded
// to 16): one 16-channel block (32-byte rows, 32-byte swizzle), one k-step per tap.
template <int CIN>
struct Cfg {
    static_assert(CIN == 96 || CIN == 16, "supported input widths");
    static constexpr unsigned ROW0 = CIN == 96 ? 128u : 32u, ROW1 = CIN == 96 ? 64u : 0u;     // bytes per pixel row
    static constexpr int KS0 = CIN == 96 ? 4 : 1, KS1 = CIN == 96 ? 2 : 0;                    // 16-channel k-steps
    static constexpr int BOX0 = CIN == 96 ? 64 : 16, BOX1 = 32;                               // TMA box widths (channels)
    static constexpr unsigned W0_TAP = C * ROW0, W1_TAP = C * ROW1;     // bytes per weight tap
    static constexpr unsigned W0_BYTES = 9 * W0_TAP, W1_BYTES = 9 * W1_TAP;
    static constexpr unsigned A0_BYTES = PX_IN * ROW0, A1_BYTES = PX_IN * ROW1, A_STAGE = A0_BYTES + A1_BYTES;
    static constexpr unsigned PAD = 1024u;                               // the dx = -1 tap of the first row reads one row before the block
    static constexpr unsigned OFF_W0 = 0, OFF_W1 = OFF_W0 + W0_BYTES, OFF_A = ((OFF_W1 + W1_BYTES + 1023u) & ~1023u) + (CIN == 96 ? 0u : PAD);
    static constexpr unsigned OFF_BAR = (OFF_A + STAGES * A_STAGE + 1023u) & ~1023u;   // full[2], empty[2], wfull, tfull[4], tempty[4]
    static constexpr unsigned OFF_TMEM = OFF_BAR + 13 * 8u;
    static constexpr unsigned OFF_PART = (OFF_TMEM + 16u + 15u) & ~15u;  // GN epilogue: [2 parity][12 warps][2 groups][mean, M2] f32
    static constexpr unsigned OFF_CB = OFF_PART + 2 * 2 * 12 * 2 * 4u;   // [96] conv bias
    static constexpr unsigned OFF_AB = OFF_CB + C * 4u;                  // [2 parity][2][96]: per-channel scale a, shift b of the board
    static constexpr unsigned SMEM_BYTES = OFF_AB + 2 * 2 * C * 4u + 1024u;   // + slack to align the base to 1024 B
};
}  // namespace cv

// What the fused GroupNorm epilogue needs (conv3x3_tc_kernel<true>); same meaning as msw_gn_act's arguments.
//
// The fp32 residual stream (res32 in, y32 out) is private to this kernel family, so it lives in HBM in the order
// the epilogue touches it -- "P8": [board][tile 2][channel third 3][8-channel chunk 4][pixel 128][8 floats].  A
// thread (= pixel) owns one 32-byte chunk per (third, chunk); the 32 lanes of a warp are 32 consecutive pixels,
// so every 256-bit load / store instruction of a warp covers 1 KB of consecutive addresses (8 full lines)
// instead of one line per lane as the pixel-major NHWC order would (32 lines per instruction: the epilogue was
// LSU-bound at 690 us per layer with it, against 240 us of MMAs).
struct ConvGnParams {
    const float *cbias, *gamma, *beta;   // [96]
    const float *res32;                  // nullable, P8 order
    float *y32;                          // nullable, P8 order
    float *pool4;                        // nullable [n][4][96]: per row-quarter sums of the fp32 output (value head's avg pool)
    float eps, drop_p, drop_scale;
    uint32_t k0, k1, call_lo, call_hi;
    const uint32_t *epoch;               // nullable
    long long sample_base;               // global index of board 0 (Dropout2d stream is keyed by the global board)
};

// float offset of (board, tile, third, chunk, pixel-in-tile) in the P8 order
__device__ __forceinline__ long long cv_p8(long long board, int half, int third, int c4, int pp)
{
    return ((((board * 2 + half) * 3 + third) * 4 + c4) * 128 + pp) * 8;
}

__device__ __forceinline__ void cv_st256(void *p, const uint32_t (&v)[8])
{
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void cv_ld256(const void *p, uint32_t (&v)[8])
{
    asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "l"(p));
}
__device__ __forceinline__ float cv_warp_sum(float v)          // fixed shuffle tree: deterministic
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// GN = false: out = conv(x) (fp16).  GN = true: out = relu(GroupNorm(conv(x) + bias) [+ res]) [* Dropout2d], the
// whole inter-convolution step of msw_gn_act fused into the epilogue (6 groups of 16 channels; statistics over
// the board = the CTA's two consecutive tiles, whose fp16-rounded conv outputs wait in registers).
// EPI (GN only): 0 = no residual (Dropout2d allowed, y32 optional), 1 = residual in, y32 out, 2 = residual in, pooled
// sums out (the last block: nothing reads its residual stream but the value head's average pool).
template <bool GN, int CIN, int EPI>
__global__ void __launch_bounds__(cv::THREADS, 1)
conv3x3_tc_kernel(const __grid_constant__ CUtensorMap map_a0, const __grid_constant__ CUtensorMap map_a1,
                  const __grid_constant__ CUtensorMap map_w0, const __grid_constant__ CUtensorMap map_w1,
                  __half *__restrict__ out, long long boards, int dbg, const __grid_constant__ ConvGnParams gp)
{
    using namespace cv;
    using K = Cfg<CIN>;
    constexpr unsigned OFF_W0 = K::OFF_W0, OFF_W1 = K::OFF_W1, OFF_A = K::OFF_A, OFF_BAR = K::OFF_BAR, OFF_TMEM = K::OFF_TMEM,
                       OFF_PART = K::OFF_PART, OFF_CB = K::OFF_CB, OFF_AB = K::OFF_AB, W0_TAP = K::W0_TAP, W1_TAP = K::W1_TAP,
                       A0_BYTES = K::A0_BYTES, A_STAGE = K::A_STAGE;
    extern __shared__ unsigned char smem_dyn[];
    const unsigned base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
    unsigned char *gen = smem_dyn + (base - smem_u32(smem_dyn));
    const unsigned bars = base + OFF_BAR;
    auto full = [&](int s) { return bars + 8u * s; };
    auto empty = [&](int s) { return bars + 8u * (2 + s); };
    const unsigned wfull = bars + 8u * 4;
    auto tfull = [&](unsigned a) { return bars + 8u * (5 + a); };
    auto tempty = [&](unsigned a) { return bars + 8u * (9 + a); };
    volatile uint32_t *s_tmem = reinterpret_cast<volatile uint32_t *>(gen + OFF_TMEM);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full(s), 1); mbar_init(empty(s), 1); }
        for (unsigned a = 0; a < ACC; ++a) { mbar_init(tfull(a), 1); mbar_init(tempty(a), 12); }
        mbar_init(wfull, 1);
        mbar_fence_init();
    }
    if (warp == 2) tmem_alloc(base + OFF_TMEM, TMEM_COLS);
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const unsigned tmem = *s_tmem;

    if (warp == 0) {
        if (elect_one()) {
        // ---- TMA producer: the nine weight taps once, then one [10 rows x 16 px x 96 ch] block per tile
        mbar_expect_tx(wfull, K::W0_BYTES + K::W1_BYTES);
        for (int t = 0; t < 9; ++t) {
            tma_load_2d(base + OFF_W0 + t * W0_TAP, &map_w0, 0, t * C, wfull);
            if (K::KS1) tma_load_2d(base + OFF_W1 + t * W1_TAP, &map_w1, K::BOX0, t * C, wfull);
        }
        // a CTA takes whole boards: tiles 2*board, 2*board + 1 back to back (the GN epilogue needs both)
        for (unsigned it = 0;; ++it) {
            const long long board = blockIdx.x + (long long)(it >> 1) * gridDim.x;
            if (board >= boards) break;
            const unsigned s = it % STAGES, ph = (it / STAGES) & 1u;
            const int n = (int)board, y0 = (int)(it & 1u) * 8;
            mbar_wait(empty(s), ph ^ 1u);
            mbar_expect_tx(full(s), A_STAGE);
            tma_load_4d(base + OFF_A + s * A_STAGE, &map_a0, 0, 0, y0 - 1, n, full(s));
            if (K::KS1) tma_load_4d(base + OFF_A + s * A_STAGE + A0_BYTES, &map_a1, K::BOX0, 0, y0 - 1, n, full(s));
        }
        }
    } else if (warp == 1) {
        // ---- MMA issuer.  idesc: D = F32, A = B = F16, K-major, M = 128, N = 96.
        constexpr unsigned idesc = (1u << 4) | ((unsigned)(C >> 3) << 17) | ((unsigned)(TILE_PX >> 4) << 24);
        mbar_wait(wfull, 0);
        for (unsigned it = 0;; ++it) {
            if (blockIdx.x + (long long)(it >> 1) * gridDim.x >= boards) break;
            const unsigned s = it % STAGES, ph = (it / STAGES) & 1u, acc = it % ACC, aph = (it / ACC) & 1u;
            mbar_wait(tempty(acc), aph ^ 1u);                     // the epilogue has drained this accumulator
            mbar_wait(full(s), ph);
            tcgen05_fence_after();
            const unsigned a0 = base + OFF_A + s * A_STAGE, a1 = a0 + A0_BYTES, d = tmem + acc * C;
            if (elect_one()) {            // the whole warp runs the loop and the waits; one elected lane issues
            unsigned accumulate = 0u;
            if (!MSW_DBG(8))
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int o = 0; o < 3; ++o) {
                    const int dxi = o == 0 ? 1 : o == 1 ? 0 : 2;           // the unmasked centre tap first
                    const int tap = dy * 3 + dxi;
                    // rows of D whose horizontal neighbour is off the board: x = 0 for dx = -1, x = 15 for dx = +1
                    const unsigned mask = dxi == 0 ? 0x00010001u : dxi == 2 ? 0x80008000u : 0u;
                    const unsigned sa0 = a0 + (unsigned)((dy * HW_W + dxi - 1) * (int)K::ROW0);
                    const unsigned sa1 = a1 + (unsigned)((dy * HW_W + dxi - 1) * (int)K::ROW1);
#pragma unroll
                    for (int k = 0; k < K::KS0; ++k) {                       // first channel block, 16 channels (32 bytes) per step
                        umma_f16_masked(d, umma_desc<K::ROW0>(sa0) + 2u * k, umma_desc<K::ROW0>(base + OFF_W0 + tap * W0_TAP) + 2u * k,
                                        idesc, accumulate, mask);
                        accumulate = 1u;
                    }
                    if constexpr (K::KS1 > 0) {
#pragma unroll
                        for (int k = 0; k < K::KS1; ++k)                     // second channel block
                            umma_f16_masked(d, umma_desc<K::ROW1>(sa1) + 2u * k,
                                            umma_desc<K::ROW1>(base + OFF_W1 + tap * W1_TAP) + 2u * k, idesc, 1u, mask);
                    }
                }
            umma_commit(empty(s));           // the smem stage is free once these MMAs have read it
            umma_commit(tfull(acc));         // ... and the accumulator is complete
            }
            __syncwarp();
        }
    } else if (warp >= 4) {
        // ---- epilogue: thread = pixel (TMEM lane q*32 + lane), each of the three warpgroups a third of the channels
        const int q = warp & 3, third = (warp - 4) >> 2;
        if constexpr (!GN) {
        for (unsigned it = 0;; ++it) {
            const long long board = blockIdx.x + (long long)(it >> 1) * gridDim.x;
            if (board >= boards) break;
            const unsigned acc = it % ACC, aph = (it / ACC) & 1u;
            mbar_wait(tfull(acc), aph);
            tcgen05_fence_after();
            uint32_t v[32];
            {
                uint32_t lo[16], hi[16];
                const unsigned taddr = tmem + ((unsigned)(q * 32) << 16) + acc * C + third * 32;
                tmem_ld16(taddr, lo);
                tmem_ld16(taddr + 16, hi);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 16; ++j) { v[j] = lo[j]; v[16 + j] = hi[j]; }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty(acc));       // the accumulator is in registers: release it
            if (MSW_DBG(1)) continue;
            __half *dst = out + (board * 256 + (it & 1u) * 128 + q * 32 + lane) * (long long)C + third * 32;
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 16) {
                uint32_t packed[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const __half2 hh = __floats2half2_rn(__uint_as_float(v[c0 + 2 * k]), __uint_as_float(v[c0 + 2 * k + 1]));
                    packed[k] = *reinterpret_cast<const uint32_t *>(&hh);
                }
                // one 256-bit store per lane: the lanes of a warp write to 32 different 128-byte lines either way
                // (pixels are 192 B apart), so the LSU cost is per instruction, not per byte
                cv_st256(dst + c0, packed);
            }
        }
        } else {
        // ---- fused GroupNorm epilogue.  Thread = pixel, its 32 channels = groups 2*third and 2*third + 1.
        const int we = warp - 4, te = tid - 128;                        // epilogue warp 0..11 = third*4 + q, thread 0..383
        float *s_part = reinterpret_cast<float *>(gen + OFF_PART);      // [parity][warp][group][mean, M2]
        float *s_cb = reinterpret_cast<float *>(gen + OFF_CB);          // conv bias
        float *s_ab = reinterpret_cast<float *>(gen + OFF_AB);          // [parity][a | b][channel]
        const int cbase = third * 32;
        const uint32_t thresh = (uint32_t)(gp.drop_p * 65536.0f);
        if (te < C) s_cb[te] = gp.cbias[te];
        asm volatile("bar.sync 1, 384;" ::: "memory");
        const float2 *cb2 = reinterpret_cast<const float2 *>(s_cb + cbase);
        for (unsigned bi = 0;; ++bi) {
            const long long board = blockIdx.x + (long long)bi * gridDim.x;
            if (board >= boards) break;
            const unsigned par = bi & 1u;
            // Dropout2d scale of channel `te` for this board (msw_gn_act's stream: Philox keyed by board and 8-channel
            // chunk).  It does not depend on the data, so it is drawn here, off the path between the two barriers.
            float sc = gp.drop_scale;
            if (EPI == 0 && te < C && gp.drop_p > 0.0f) {
                uint32_t w[4];
                const long long gb = gp.sample_base + board;
                philox4x32_10(gp.k0, gp.k1 ^ 0x44524f50u, (uint32_t)gb, (uint32_t)(gb >> 32) ^ (uint32_t)(te >> 3), gp.call_lo,
                              gp.call_hi + (gp.epoch ? *gp.epoch : 0u), w);
                const int k = te & 7;
                const uint32_t u16 = (w[k >> 1] >> (16 * (k & 1))) & 0xFFFFu;
                if (u16 < thresh) sc = 0.0f;
            }
            uint32_t h[2][16];                       // fp16-rounded conv output of both tiles (the reference's rounding point)
            // One-pass statistics of v = x + bias, shifted by a value of the warp's own data (no cancellation in
            // S2 - S1^2/n): per thread S1 = sum (v - shift), S2 = sum (v - shift)^2 for its two groups.
            float shift0 = 0.0f, shift1 = 0.0f, s1a = 0.0f, s2a = 0.0f, s1b = 0.0f, s2b = 0.0f;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const unsigned it = 2u * bi + half, acc = it % ACC, aph = (it / ACC) & 1u;
                if (EPI != 0)     // the 16 KB of residual stream this warpgroup will read for this tile: one line per thread on its way to L2
                    asm volatile("prefetch.global.L2 [%0];" :: "l"(gp.res32 + cv_p8(board, half, third, 0, 0) + (q * 32 + lane) * 32));
                mbar_wait(tfull(acc), aph);
                tcgen05_fence_after();
                uint32_t lo[16], hi[16];
                const unsigned taddr = tmem + ((unsigned)(q * 32) << 16) + acc * C + third * 32;
                tmem_ld16(taddr, lo);
                tmem_ld16(taddr + 16, hi);
                tmem_wait_ld();
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty(acc));
                if (MSW_DBG(16)) continue;
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) {
                    const uint32_t *src = jj < 8 ? lo : hi;
                    const __half2 hh = __floats2half2_rn(__uint_as_float(src[(2 * jj) & 15]), __uint_as_float(src[(2 * jj + 1) & 15]));
                    h[half][jj] = *reinterpret_cast<const uint32_t *>(&hh);
                    const float2 f = __half22float2(hh), cb = cb2[jj];
                    const float v0 = f.x + cb.x, v1 = f.y + cb.y;
                    if (half == 0 && jj == 0) shift0 = __shfl_sync(0xffffffffu, v0, 0);
                    if (half == 0 && jj == 8) shift1 = __shfl_sync(0xffffffffu, v0, 0);
                    if (jj < 8) {
                        const float d0 = v0 - shift0, d1 = v1 - shift0;
                        s1a += d0 + d1;
                        s2a = fmaf(d0, d0, fmaf(d1, d1, s2a));
                    } else {
                        const float d0 = v0 - shift1, d1 = v1 - shift1;
                        s1b += d0 + d1;
                        s2b = fmaf(d0, d0, fmaf(d1, d1, s2b));
                    }
                }
            }
            if (MSW_DBG(16)) continue;
            // the warp's (mean, M2) over its 1,024 values per group; the board's statistics are merged from the four
            // row-owning warps of a channel third in a fixed order (Chan et al.)
            s1a = cv_warp_sum(s1a); s2a = cv_warp_sum(s2a);
            s1b = cv_warp_sum(s1b); s2b = cv_warp_sum(s2b);
            if (lane == 0) {
                float *dst = s_part + (par * 12 + we) * 4;
                dst[0] = shift0 + s1a * (1.0f / 1024.0f); dst[1] = s2a - s1a * s1a * (1.0f / 1024.0f);
                dst[2] = shift1 + s1b * (1.0f / 1024.0f); dst[3] = s2b - s1b * s1b * (1.0f / 1024.0f);
            }
            if (!MSW_DBG(2)) asm volatile("bar.sync 1, 384;" ::: "memory");
            if (te < C) {
                // one thread per channel folds statistics, affine, conv bias and the Dropout2d scale into y = a*x + b
                const int c = te, gsel = (c >> 4) & 1, w4 = (c >> 5) * 4;
                float na = 0.0f, mg = 0.0f, m2 = 0.0f;
#pragma unroll
                for (int qq = 0; qq < 4; ++qq) {
                    const float *src = s_part + (par * 12 + w4 + qq) * 4 + 2 * gsel;
                    const float nn = na + 1024.0f, delta = src[0] - mg, w = 1024.0f / nn;
                    mg = fmaf(delta, w, mg);
                    m2 += src[1] + delta * delta * (na * w);
                    na = nn;
                }
                const float rg = rsqrtf(m2 * (1.0f / 4096.0f) + gp.eps);       // biased variance, eps as torch
                const float a = gp.gamma[c] * rg;
                s_ab[(par * 2 + 0) * C + c] = a * sc;
                s_ab[(par * 2 + 1) * C + c] = fmaf(s_cb[c] - mg, a, gp.beta[c]) * sc;
            }
            if (!MSW_DBG(2)) asm volatile("bar.sync 1, 384;" ::: "memory");
            // ---- normalise, (+ residual), ReLU, store: chunk by chunk (8 channels), both tiles per chunk
            const float4 *a4 = reinterpret_cast<const float4 *>(s_ab + (par * 2 + 0) * C + cbase);
            const float4 *b4 = reinterpret_cast<const float4 *>(s_ab + (par * 2 + 1) * C + cbase);
            const int pp = q * 32 + lane;
            uint32_t rnext[8];                       // residual values of the next (chunk, tile): loaded one step ahead
            if (EPI != 0) cv_ld256(gp.res32 + cv_p8(board, 0, third, 0, pp), rnext);
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 8) {
                const float4 aa0 = a4[c0 >> 2], aa1 = a4[(c0 >> 2) + 1], bb0 = b4[c0 >> 2], bb1 = b4[(c0 >> 2) + 1];
                const float av[8] = {aa0.x, aa0.y, aa0.z, aa0.w, aa1.x, aa1.y, aa1.z, aa1.w};
                const float bv[8] = {bb0.x, bb0.y, bb0.z, bb0.w, bb1.x, bb1.y, bb1.z, bb1.w};
                float ps[8];                         // EPI 2: this thread's two pixels summed, per channel
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    uint32_t rr[8];
                    if (EPI != 0) {
#pragma unroll
                        for (int k = 0; k < 8; ++k) rr[k] = rnext[k];
                        if (half == 0) cv_ld256(gp.res32 + cv_p8(board, 1, third, c0 >> 3, pp), rnext);
                        else if (c0 < 24) cv_ld256(gp.res32 + cv_p8(board, 0, third, (c0 >> 3) + 1, pp), rnext);
                    }
                    uint32_t o[8];
#pragma unroll
                    for (int j = 0; j < 8; j += 2) {
                        const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&h[half][(c0 + j) >> 1]));
                        float v0 = fmaf(f.x, av[j], bv[j]), v1 = fmaf(f.y, av[j + 1], bv[j + 1]);
                        if (EPI != 0) { v0 += __uint_as_float(rr[j]); v1 += __uint_as_float(rr[j + 1]); }
                        v0 = fmaxf(v0, 0.0f); v1 = fmaxf(v1, 0.0f);
                        o[j] = __float_as_uint(v0);
                        o[j + 1] = __float_as_uint(v1);
                        if (EPI == 2) {
                            ps[j] = half == 0 ? v0 : ps[j] + v0;
                            ps[j + 1] = half == 0 ? v1 : ps[j + 1] + v1;
                        }
                    }
                    if (EPI != 2 && gp.y32 && !MSW_DBG(1)) cv_st256(gp.y32 + cv_p8(board, half, third, c0 >> 3, pp), o);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const __half2 hh = __floats2half2_rn(__uint_as_float(o[2 * k]), __uint_as_float(o[2 * k + 1]));
                        h[half][(c0 >> 1) + k] = *reinterpret_cast<const uint32_t *>(&hh);     // reuse the slot for the output
                    }
                }
                if (EPI == 2) {
                    // warp sum of 8 channels over the 32 lanes in 9 shuffles (fixed butterfly: deterministic): each
                    // step halves the number of channels a lane carries; lane L ends with channel bit4*4 + bit3*2 + bit2
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
                    if ((lane & 3) == 0)
                        gp.pool4[(board * 4 + q) * C + cbase + c0 + (b4s ? 4 : 0) + (b3s ? 2 : 0) + (b2s ? 1 : 0)] = a3;
                }
            }
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const long long px = board * 256 + half * 128 + pp;
#pragma unroll
                for (int c0 = 0; c0 < 32; c0 += 16) {
                    uint32_t packed[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) packed[k] = h[half][(c0 >> 1) + k];
                    if (!MSW_DBG(1)) cv_st256(out + px * C + cbase + c0, packed);
                }
            }
        }
        }
    }

    tcgen05_fence_before();
    __syncthreads();
    if (warp == 2) {
        tcgen05_fence_after();
        tmem_dealloc(tmem, TMEM_COLS);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// 128 output channels: one board per CTA pair (2-CTA cluster, tcgen05 cta_group::2, M = 256, N = 128).
//
// At C = 128 the nine [128 x 128] weight taps take 288 KB, more than a CTA's shared memory, so each CTA of the pair
// holds the nine taps of HALF the output channels (rank r: [64r, 64r + 64), 147,456 B) and stages tile r of the
// board (image rows 8r .. 8r + 7, i.e. input rows 8r - 1 .. 8r + 8: the same 4-D TMA box as above).  The leader
// (rank 0) issues one cta_group::2 MMA per tap and k-step for both tiles (9 taps x 8 k-steps = 72 per board); A
// rows 128 .. 255 are the peer's tile, B's 64 + 64 rows the two weight halves, and each CTA's TMEM receives its own
// 128 pixels x all 128 output channels.  Taps, shifted descriptors and the disable-output-lane masks are those of
// conv3x3_tc_kernel, the mask covering the 256 rows of the pair.  K = 128 = two 64-channel blocks (128-byte rows,
// 128-byte swizzle; both through the same tensor map); the stem (CIN = 16) is as above.
//
// GroupNorm statistics of a board span both tiles.  Every epilogue warp writes its (mean, M2) of its two groups
// into its own CTA's exchange area AND the partner's (st.shared::cluster), then arrives on the partner's xfull
// barrier; both CTAs then merge the same 2 x 16 partials in the same order, so they fold bit-identical a and b.  No
// cluster barrier inside the loop: the producer and MMA warps never wait on an epilogue's statistics.
//
// Shared memory per CTA (CIN = 128; 232,064 of 232,448 B), from a 1024-byte aligned base:
//        0  W0  [9 taps][64 co][64 ch]  128-byte swizzle     73,728
//   73,728  W1  [9 taps][64 co][64 ch]  (channels 64..127)   73,728
//  147,456  A   [2 stages][2 blocks][160 px][64 ch]          81,920
//  229,376  barriers full[2] empty[2] wfull tfull[4] tempty[4] xfull[2], TMEM address   128
//  229,504  X   [2 parity][2 tile][16 warps][mean0, M2_0, mean1, M2_1] f32               1,024
//  230,528  conv bias [128] f32                                                          512
//  231,040  a | b [2][128] f32                                                           1,024
// Roles: warp 0 TMA producer (both CTAs), warp 1 MMA issuer (leader), warp 2 TMEM allocation (both), warps 4-19
// epilogue (thread = pixel of the CTA's tile, warpgroup g = channels [32g, 32g + 32): groups 2g and 2g + 1).
namespace cvp {
constexpr int C = 128, HALF = 64, HW_W = 16, TILE_PX = 128, PX_IN = 160;
constexpr int THREADS = 640, EPI_WARPS = 16, STAGES = 2, ACC = 4, TMEM_COLS = 512;    // 4 x 128 accumulator columns

template <int CIN>
struct Cfg {
    static_assert(CIN == 128 || CIN == 16, "supported input widths");
    static constexpr unsigned ROW0 = CIN == 128 ? 128u : 32u, ROW1 = CIN == 128 ? 128u : 0u;   // bytes per pixel row
    static constexpr int KS0 = CIN == 128 ? 4 : 1, KS1 = CIN == 128 ? 4 : 0;                   // 16-channel k-steps
    static constexpr int BOX0 = CIN == 128 ? 64 : 16;                                          // channels per block
    static constexpr unsigned W0_TAP = HALF * ROW0, W1_TAP = HALF * ROW1;                      // this CTA's rows of a tap
    static constexpr unsigned W0_BYTES = 9 * W0_TAP, W1_BYTES = 9 * W1_TAP;
    static constexpr unsigned A0_BYTES = PX_IN * ROW0, A_STAGE = A0_BYTES + PX_IN * ROW1;
    // the stem keeps conv3x3_tc_kernel's 1 KB in front of its activation ring; at CIN = 128 the first tap's read
    // of one row before a stage lands in the weights, in rows the mask switches off
    static constexpr unsigned OFF_W0 = 0, OFF_W1 = W0_BYTES, OFF_A = W0_BYTES + W1_BYTES + (CIN == 128 ? 0u : 1024u);
    static constexpr unsigned OFF_BAR = OFF_A + STAGES * A_STAGE;
    static constexpr unsigned OFF_TMEM = OFF_BAR + 15 * 8u;
    static constexpr unsigned OFF_X = OFF_BAR + 128u;
    static constexpr unsigned OFF_CB = OFF_X + 2 * 2 * EPI_WARPS * 4 * 4u;
    static constexpr unsigned OFF_AB = OFF_CB + C * 4u;
    static constexpr unsigned SMEM_BYTES = OFF_AB + 2 * C * 4u;
    static_assert(OFF_A % 1024 == 0 && A0_BYTES % 1024 == 0 && A_STAGE % 1024 == 0 && W0_TAP % 1024 == 0, "swizzle atoms");
    static_assert(SMEM_BYTES <= 232448, "shared memory of one CTA");
};
}  // namespace cvp

// float offset of (board, tile, quarter, chunk, pixel-in-tile) in the C = 128 P8 order
__device__ __forceinline__ long long cvp_p8(long long board, int tile, int quarter, int c4, int pp)
{
    return ((((board * 2 + tile) * 4 + quarter) * 4 + c4) * 128 + pp) * 8;
}

// GN / CIN / EPI as conv3x3_tc_kernel; pool4 is [n][tile 2 x row quarter 4][128].
template <bool GN, int CIN, int EPI>
__global__ void __launch_bounds__(cvp::THREADS, 1)
conv3x3_pair_kernel(const __grid_constant__ CUtensorMap map_a0, const __grid_constant__ CUtensorMap map_a1,
                    const __grid_constant__ CUtensorMap map_w0, const __grid_constant__ CUtensorMap map_w1,
                    __half *__restrict__ out, long long boards, const __grid_constant__ ConvGnParams gp)
{
    using namespace cvp;
    using K = Cfg<CIN>;
    constexpr unsigned OFF_A = K::OFF_A, W0_TAP = K::W0_TAP, W1_TAP = K::W1_TAP, A0_BYTES = K::A0_BYTES, A_STAGE = K::A_STAGE;
    extern __shared__ __align__(1024) unsigned char smem_pair[];
    const unsigned base = smem_u32(smem_pair);
    if (base & 1023u) {                  // the layout has no room to realign; uniform over the grid
        if (threadIdx.x == 0 && blockIdx.x == 0) printf("conv3x3_pair_kernel: dynamic shared memory is not 1024-byte aligned\n");
        return;
    }
    const unsigned bars = base + K::OFF_BAR;
    auto full = [&](unsigned s) { return bars + 8u * s; };
    auto empty = [&](unsigned s) { return bars + 8u * (2 + s); };
    const unsigned wfull = bars + 8u * 4;
    auto tfull = [&](unsigned a) { return bars + 8u * (5 + a); };
    auto tempty = [&](unsigned a) { return bars + 8u * (9 + a); };
    auto xfull = [&](unsigned p) { return bars + 8u * (13 + p); };
    volatile uint32_t *s_tmem = reinterpret_cast<volatile uint32_t *>(smem_pair + K::OFF_TMEM);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned rank = cluster_ctarank(), peer = rank ^ 1u;
    const long long board0 = blockIdx.x >> 1, bstride = gridDim.x >> 1;     // the pair's boards: board0 + i * bstride
    if (tid == 0) {
        for (unsigned s = 0; s < STAGES; ++s) { mbar_init(full(s), 2); mbar_init(empty(s), 1); }   // full: both producers
        for (unsigned a = 0; a < ACC; ++a) { mbar_init(tfull(a), 1); mbar_init(tempty(a), 2 * EPI_WARPS); }
        mbar_init(wfull, 2);
        for (unsigned p = 0; p < 2; ++p) mbar_init(xfull(p), EPI_WARPS);    // the partner's epilogue warps
        mbar_fence_init();
    }
    if (warp == 2) tmem_alloc_pair(base + K::OFF_TMEM, TMEM_COLS);
    tcgen05_fence_before();
    cluster_sync();                      // both CTAs' barriers are initialised before anyone arrives on them
    tcgen05_fence_after();
    const unsigned tmem = *s_tmem;

    if (warp == 0) {
        if (elect_one()) {
        // ---- TMA producer: this CTA's 64 output channels of the nine taps once, then tile `rank` of every board;
        // completion is counted on the leader's barriers (the MMA issuer's)
        const unsigned wbar = mapa_shared(wfull, 0u);
        const int wrow = (int)rank * HALF;
        mbar_expect_tx_cluster(wbar, K::W0_BYTES + K::W1_BYTES);
        for (int t = 0; t < 9; ++t) {
            tma_load_2d_pair(base + K::OFF_W0 + t * W0_TAP, &map_w0, 0, t * C + wrow, wbar);
            if (K::KS1) tma_load_2d_pair(base + K::OFF_W1 + t * W1_TAP, &map_w1, K::BOX0, t * C + wrow, wbar);
        }
        for (unsigned it = 0;; ++it) {
            const long long board = board0 + (long long)it * bstride;
            if (board >= boards) break;
            const unsigned s = it % STAGES, ph = (it / STAGES) & 1u;
            mbar_wait(empty(s), ph ^ 1u);
            const unsigned fbar = mapa_shared(full(s), 0u);
            mbar_expect_tx_cluster(fbar, A_STAGE);
            tma_load_4d_pair(base + OFF_A + s * A_STAGE, &map_a0, 0, 0, 8 * (int)rank - 1, (int)board, fbar);
            if (K::KS1) tma_load_4d_pair(base + OFF_A + s * A_STAGE + A0_BYTES, &map_a1, K::BOX0, 0, 8 * (int)rank - 1, (int)board, fbar);
        }
        }
    } else if (warp == 1 && rank == 0) {
        // ---- MMA issuer.  idesc: D = F32, A = B = F16, K-major, M = 256 (the pair), N = 128.
        constexpr unsigned idesc = (1u << 4) | ((unsigned)(C >> 3) << 17) | ((unsigned)((2 * TILE_PX) >> 4) << 24);
        mbar_wait(wfull, 0);
        for (unsigned it = 0;; ++it) {
            if (board0 + (long long)it * bstride >= boards) break;
            const unsigned s = it % STAGES, ph = (it / STAGES) & 1u, acc = it % ACC, aph = (it / ACC) & 1u;
            mbar_wait_cluster(tempty(acc), aph ^ 1u);            // both CTAs' epilogues have drained this accumulator
            mbar_wait_cluster(full(s), ph);                      // both tiles have landed
            tcgen05_fence_after();
            const unsigned a0 = base + OFF_A + s * A_STAGE, a1 = a0 + A0_BYTES, d = tmem + acc * C;
            if (elect_one()) {
            unsigned accumulate = 0u;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int o = 0; o < 3; ++o) {
                    const int dxi = o == 0 ? 1 : o == 1 ? 0 : 2;           // the unmasked centre tap first
                    const int tap = dy * 3 + dxi;
                    const unsigned mask = dxi == 0 ? 0x00010001u : dxi == 2 ? 0x80008000u : 0u;
                    const unsigned sa0 = a0 + (unsigned)((dy * HW_W + dxi - 1) * (int)K::ROW0);
                    const unsigned sa1 = a1 + (unsigned)((dy * HW_W + dxi - 1) * (int)K::ROW1);
#pragma unroll
                    for (int k = 0; k < K::KS0; ++k) {
                        umma_f16_masked_pair(d, umma_desc<K::ROW0>(sa0) + 2u * k,
                                             umma_desc<K::ROW0>(base + K::OFF_W0 + tap * W0_TAP) + 2u * k, idesc, accumulate, mask);
                        accumulate = 1u;
                    }
                    if constexpr (K::KS1 > 0) {
#pragma unroll
                        for (int k = 0; k < K::KS1; ++k)
                            umma_f16_masked_pair(d, umma_desc<K::ROW1>(sa1) + 2u * k,
                                                 umma_desc<K::ROW1>(base + K::OFF_W1 + tap * W1_TAP) + 2u * k, idesc, 1u, mask);
                    }
                }
            umma_commit_pair(empty(s));          // both CTAs' stage s is free once these MMAs have read it
            umma_commit_pair(tfull(acc));        // ... and both halves of the accumulator are complete
            }
            __syncwarp();
        }
    } else if (warp >= 4) {
        const int we = warp - 4, q = warp & 3, wg = we >> 2, cbase = wg * 32, te = tid - 128, pp = q * 32 + lane;
        if constexpr (!GN) {
        for (unsigned it = 0;; ++it) {
            const long long board = board0 + (long long)it * bstride;
            if (board >= boards) break;
            const unsigned acc = it % ACC, aph = (it / ACC) & 1u;
            mbar_wait(tfull(acc), aph);
            tcgen05_fence_after();
            uint32_t lo[16], hi[16];
            const unsigned taddr = tmem + ((unsigned)(q * 32) << 16) + acc * C + cbase;
            tmem_ld16(taddr, lo);
            tmem_ld16(taddr + 16, hi);
            tmem_wait_ld();
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(mapa_shared(tempty(acc), 0u));
            __half *dst = out + (board * 256 + rank * 128 + pp) * (long long)C + cbase;
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 16) {
                const uint32_t *src = c0 == 0 ? lo : hi;
                uint32_t packed[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const __half2 hh = __floats2half2_rn(__uint_as_float(src[2 * k]), __uint_as_float(src[2 * k + 1]));
                    packed[k] = *reinterpret_cast<const uint32_t *>(&hh);
                }
                cv_st256(dst + c0, packed);
            }
        }
        } else {
        float *s_x = reinterpret_cast<float *>(smem_pair + K::OFF_X);    // [parity][tile][warp][mean0, M2_0, mean1, M2_1]
        float *s_cb = reinterpret_cast<float *>(smem_pair + K::OFF_CB);
        float *s_ab = reinterpret_cast<float *>(smem_pair + K::OFF_AB);  // [a | b][channel]
        const uint32_t thresh = (uint32_t)(gp.drop_p * 65536.0f);
        if (te < C) s_cb[te] = gp.cbias[te];
        asm volatile("bar.sync 1, 512;" ::: "memory");
        const float2 *cb2 = reinterpret_cast<const float2 *>(s_cb + cbase);
        const unsigned x_peer = mapa_shared(base + K::OFF_X, peer);
        for (unsigned bi = 0;; ++bi) {
            const long long board = board0 + (long long)bi * bstride;
            if (board >= boards) break;
            const unsigned par = bi & 1u, acc = bi % ACC, aph = (bi / ACC) & 1u;
            float sc = gp.drop_scale;            // Dropout2d: msw_gn_act's stream, keyed by global board and 8-channel chunk
            if (EPI == 0 && te < C && gp.drop_p > 0.0f) {
                uint32_t w[4];
                const long long gb = gp.sample_base + board;
                philox4x32_10(gp.k0, gp.k1 ^ 0x44524f50u, (uint32_t)gb, (uint32_t)(gb >> 32) ^ (uint32_t)(te >> 3), gp.call_lo,
                              gp.call_hi + (gp.epoch ? *gp.epoch : 0u), w);
                const int k = te & 7;
                const uint32_t u16 = (w[k >> 1] >> (16 * (k & 1))) & 0xFFFFu;
                if (u16 < thresh) sc = 0.0f;
            }
            if (EPI != 0)     // the 16 KB of residual stream this warpgroup reads for this tile: one line per thread
                asm volatile("prefetch.global.L2 [%0];" :: "l"(gp.res32 + cvp_p8(board, (int)rank, wg, 0, 0) + pp * 32));
            mbar_wait(tfull(acc), aph);
            tcgen05_fence_after();
            uint32_t lo[16], hi[16];
            const unsigned taddr = tmem + ((unsigned)(q * 32) << 16) + acc * C + cbase;
            tmem_ld16(taddr, lo);
            tmem_ld16(taddr + 16, hi);
            tmem_wait_ld();
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(mapa_shared(tempty(acc), 0u));
            uint32_t h[16];                      // fp16-rounded conv output (the reference's rounding point)
            float shift0 = 0.0f, shift1 = 0.0f, s1a = 0.0f, s2a = 0.0f, s1b = 0.0f, s2b = 0.0f;
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
                const uint32_t *src = jj < 8 ? lo : hi;
                const __half2 hh = __floats2half2_rn(__uint_as_float(src[(2 * jj) & 15]), __uint_as_float(src[(2 * jj + 1) & 15]));
                h[jj] = *reinterpret_cast<const uint32_t *>(&hh);
                const float2 f = __half22float2(hh), cb = cb2[jj];
                const float v0 = f.x + cb.x, v1 = f.y + cb.y;
                if (jj == 0) shift0 = __shfl_sync(0xffffffffu, v0, 0);
                if (jj == 8) shift1 = __shfl_sync(0xffffffffu, v0, 0);
                if (jj < 8) {
                    const float d0 = v0 - shift0, d1 = v1 - shift0;
                    s1a += d0 + d1;
                    s2a = fmaf(d0, d0, fmaf(d1, d1, s2a));
                } else {
                    const float d0 = v0 - shift1, d1 = v1 - shift1;
                    s1b += d0 + d1;
                    s2b = fmaf(d0, d0, fmaf(d1, d1, s2b));
                }
            }
            // the warp's (mean, M2) of its 512 values per group, into both CTAs' exchange areas
            s1a = cv_warp_sum(s1a); s2a = cv_warp_sum(s2a);
            s1b = cv_warp_sum(s1b); s2b = cv_warp_sum(s2b);
            if (lane == 0) {
                const float4 st = make_float4(shift0 + s1a * (1.0f / 512.0f), s2a - s1a * s1a * (1.0f / 512.0f),
                                              shift1 + s1b * (1.0f / 512.0f), s2b - s1b * s1b * (1.0f / 512.0f));
                const unsigned slot = ((par * 2 + rank) * EPI_WARPS + we) * 16u;
                *reinterpret_cast<float4 *>(smem_pair + K::OFF_X + slot) = st;
                st_shared_cluster_v4(x_peer + slot, st);
                mbar_arrive_cluster(mapa_shared(xfull(par), peer));
            }
            asm volatile("bar.sync 1, 512;" ::: "memory");
            if (te < C) {
                // one thread per channel: the board's statistics from tile 0's then tile 1's four warps (Chan et al.,
                // the same order in both CTAs), folded with the affine, the conv bias and the Dropout2d scale
                mbar_wait_cluster(xfull(par), (bi >> 1) & 1u);
                const int c = te, gsel = (c >> 4) & 1, w4 = (c >> 5) * 4;
                float na = 0.0f, mg = 0.0f, m2 = 0.0f;
#pragma unroll
                for (int t = 0; t < 2; ++t)
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq) {
                        const float *src = s_x + ((par * 2 + t) * EPI_WARPS + w4 + qq) * 4 + 2 * gsel;
                        const float nn = na + 512.0f, delta = src[0] - mg, w = 512.0f / nn;
                        mg = fmaf(delta, w, mg);
                        m2 += src[1] + delta * delta * (na * w);
                        na = nn;
                    }
                const float rg = rsqrtf(m2 * (1.0f / 4096.0f) + gp.eps);
                const float a = gp.gamma[c] * rg;
                s_ab[c] = a * sc;
                s_ab[C + c] = fmaf(s_cb[c] - mg, a, gp.beta[c]) * sc;
            }
            asm volatile("bar.sync 1, 512;" ::: "memory");
            // ---- normalise, (+ residual), ReLU, store: 8 channels at a time
            const float4 *a4 = reinterpret_cast<const float4 *>(s_ab + cbase);
            const float4 *b4 = reinterpret_cast<const float4 *>(s_ab + C + cbase);
            uint32_t rnext[8];
            if (EPI != 0) cv_ld256(gp.res32 + cvp_p8(board, (int)rank, wg, 0, pp), rnext);
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 8) {
                const float4 aa0 = a4[c0 >> 2], aa1 = a4[(c0 >> 2) + 1], bb0 = b4[c0 >> 2], bb1 = b4[(c0 >> 2) + 1];
                const float av[8] = {aa0.x, aa0.y, aa0.z, aa0.w, aa1.x, aa1.y, aa1.z, aa1.w};
                const float bv[8] = {bb0.x, bb0.y, bb0.z, bb0.w, bb1.x, bb1.y, bb1.z, bb1.w};
                uint32_t rr[8];
                if (EPI != 0) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) rr[k] = rnext[k];
                    if (c0 < 24) cv_ld256(gp.res32 + cvp_p8(board, (int)rank, wg, (c0 >> 3) + 1, pp), rnext);
                }
                uint32_t o[8];
#pragma unroll
                for (int j = 0; j < 8; j += 2) {
                    const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&h[(c0 + j) >> 1]));
                    float v0 = fmaf(f.x, av[j], bv[j]), v1 = fmaf(f.y, av[j + 1], bv[j + 1]);
                    if (EPI != 0) { v0 += __uint_as_float(rr[j]); v1 += __uint_as_float(rr[j + 1]); }
                    o[j] = __float_as_uint(fmaxf(v0, 0.0f));
                    o[j + 1] = __float_as_uint(fmaxf(v1, 0.0f));
                }
                if (EPI != 2 && gp.y32) cv_st256(gp.y32 + cvp_p8(board, (int)rank, wg, c0 >> 3, pp), o);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const __half2 hh = __floats2half2_rn(__uint_as_float(o[2 * k]), __uint_as_float(o[2 * k + 1]));
                    h[(c0 >> 1) + k] = *reinterpret_cast<const uint32_t *>(&hh);
                }
                if (EPI == 2) {
                    // warp sum of 8 channels over the 32 lanes (pixels), the fixed butterfly of conv3x3_tc_kernel
                    const bool b4s = lane & 16, b3s = lane & 8, b2s = lane & 4;
                    float a1[4], a2[2], a3;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float lo4 = __uint_as_float(o[i]), hi4 = __uint_as_float(o[4 + i]);
                        a1[i] = (b4s ? hi4 : lo4) + __shfl_xor_sync(0xffffffffu, b4s ? lo4 : hi4, 16);
                    }
#pragma unroll
                    for (int i = 0; i < 2; ++i)
                        a2[i] = (b3s ? a1[2 + i] : a1[i]) + __shfl_xor_sync(0xffffffffu, b3s ? a1[i] : a1[2 + i], 8);
                    a3 = (b2s ? a2[1] : a2[0]) + __shfl_xor_sync(0xffffffffu, b2s ? a2[0] : a2[1], 4);
                    a3 += __shfl_xor_sync(0xffffffffu, a3, 2);
                    a3 += __shfl_xor_sync(0xffffffffu, a3, 1);
                    if ((lane & 3) == 0)
                        gp.pool4[(board * 8 + rank * 4 + q) * C + cbase + c0 + (b4s ? 4 : 0) + (b3s ? 2 : 0) + (b2s ? 1 : 0)] = a3;
                }
            }
            __half *dst = out + (board * 256 + rank * 128 + pp) * (long long)C + cbase;
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 16) {
                uint32_t packed[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) packed[k] = h[(c0 >> 1) + k];
                cv_st256(dst + c0, packed);
            }
        }
        }
    }

    tcgen05_fence_before();
    cluster_sync();                      // neither CTA leaves (or frees TMEM) while its partner may still signal it
    if (warp == 2) {
        tcgen05_fence_after();
        tmem_dealloc_pair(tmem, TMEM_COLS);
    }
}

}  // namespace msw

template <bool GN, int CIN, int EPI>
static int conv_launch_t(const CUtensorMap &ma0, const CUtensorMap &ma1, const CUtensorMap &mw0, const CUtensorMap &mw1, void *y16,
                         int64_t n, int dbg, const msw::ConvGnParams &gp, int max_ctas, cudaStream_t stream)
{
    using namespace msw;
    using K = cv::Cfg<CIN>;
    MSW_SET_MAX_SMEM((conv3x3_tc_kernel<GN, CIN, EPI>), K::SMEM_BYTES);
    int sms = sm_count();
    if (max_ctas > 0 && max_ctas < sms) sms = max_ctas;             // caller shares the GPU with a concurrent launch
    const long long grid = n < sms ? n : sms;                       // persistent: whole boards per CTA
    conv3x3_tc_kernel<GN, CIN, EPI><<<(unsigned)grid, cv::THREADS, K::SMEM_BYTES, stream>>>(ma0, ma1, mw0, mw1, (__half *)y16,
                                                                                       (long long)n, dbg, gp);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

// The CTA-pair kernel: clusters of 2, one board per cluster at a time, at most one cluster per two SMs (the
// launch's grid cap is rounded down to an even count).
template <bool GN, int CIN, int EPI>
static int conv_pair_launch_t(const CUtensorMap &ma0, const CUtensorMap &ma1, const CUtensorMap &mw0, const CUtensorMap &mw1,
                              void *y16, int64_t n, const msw::ConvGnParams &gp, int max_ctas, cudaStream_t stream)
{
    using namespace msw;
    using K = cvp::Cfg<CIN>;
    MSW_SET_MAX_SMEM((conv3x3_pair_kernel<GN, CIN, EPI>), K::SMEM_BYTES);
    int sms = sm_count();
    if (max_ctas > 0 && max_ctas < sms) sms = max_ctas;
    const long long pairs_max = sms / 2 > 0 ? sms / 2 : 1;
    const long long pairs = n < pairs_max ? n : pairs_max;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(2 * pairs), 1, 1);
    cfg.blockDim = dim3(cvp::THREADS, 1, 1);
    cfg.dynamicSmemBytes = K::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    MSW_CUDA_TRY(cudaLaunchKernelEx(&cfg, conv3x3_pair_kernel<GN, CIN, EPI>, ma0, ma1, mw0, mw1, (__half *)y16, (long long)n, gp));
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

// Shared host side of msw_conv3x3 / msw_conv3x3_gn: argument checks, the four tensor maps, the launch.
// C = 96 (Cin 96 or 16): conv3x3_tc_kernel, one CTA per board; C = 128 (Cin 128 or 16): conv3x3_pair_kernel.
static int conv_launch(const char *who, const void *x16, const void *w_taps16, void *y16, int64_t n, int32_t H, int32_t W,
                       int32_t Cin, int32_t C, const msw::ConvGnParams *gn, int max_ctas, void *stream)
{
    using namespace msw;
    if (!x16 || !w_taps16 || !y16) return fail(MSW_ERR_NULL, "%s: NULL pointer", who);
    if (H != 16 || W != 16 || (C != cv::C && C != cvp::C) || (Cin != C && Cin != 16))
        return fail(MSW_ERR_BAD_SHAPE, "%s: only 16x16 boards, 96 or 128 output channels and as many or 16 input channels (got %dx%d, %d -> %d)",
                    who, H, W, Cin, C);
    if (n < 0 || n > 0x3fffffffLL) return fail(MSW_ERR_BAD_SHAPE, "%s: n=%lld", who, (long long)n);
    if ((((uintptr_t)x16 | (uintptr_t)w_taps16 | (uintptr_t)y16) & 31u) != 0)
        return fail(MSW_ERR_ALIGN, "%s: tensors must be 32-byte aligned", who);
    if (n == 0) return MSW_OK;
    if (!tensor_map_encoder_available()) return fail(MSW_ERR_ARG, "%s: cuTensorMapEncodeTiled is not available", who);
    const bool pair = C == cvp::C;
    // first channel block: 64 channels / 128-byte swizzle (Cin = 96, 128) or all 16 channels / 32-byte swizzle (Cin = 16);
    // second block: 32 channels / 64-byte swizzle (Cin = 96), channels 64..127 through the first block's maps (Cin = 128)
    const cuuint32_t b0 = Cin == 16 ? 16u : 64u;
    const CUtensorMapSwizzle sw0 = Cin == 16 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B;
    // weight rows per tap and CTA: all C output channels, or half of them on a CTA pair
    const cuuint32_t wrows = pair ? (cuuint32_t)cvp::HALF : (cuuint32_t)C;
    CUtensorMap ma0, ma1, mw0, mw1;
    {
        // activation [n][16][16][Cin] fp16: dims innermost first
        const cuuint64_t dims[4] = {(cuuint64_t)Cin, 16, 16, (cuuint64_t)n};
        const cuuint64_t strides[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)Cin * 2 * 16, (cuuint64_t)Cin * 2 * 256};
        const cuuint32_t box0[4] = {b0, 16, cv::ROWS_IN, 1}, box1[4] = {32, 16, cv::ROWS_IN, 1};
        const CUresult r0 = encode_tiled(&ma0, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, x16, dims, strides, box0, sw0);
        const CUresult r1 = Cin == 96 ? encode_tiled(&ma1, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, x16, dims, strides, box1, CU_TENSOR_MAP_SWIZZLE_64B)
                                      : CUDA_SUCCESS;
        if (r0 != CUDA_SUCCESS || r1 != CUDA_SUCCESS)
            return fail(MSW_ERR_ARG, "%s: activation tensor map failed (%d, %d)", who, (int)r0, (int)r1);
        if (Cin != 96) ma1 = ma0;
    }
    {
        // weights [9 taps * C co][Cin] fp16
        const cuuint64_t dims[2] = {(cuuint64_t)Cin, (cuuint64_t)9 * C};
        const cuuint64_t strides[1] = {(cuuint64_t)Cin * 2};
        const cuuint32_t box0[2] = {b0, wrows}, box1[2] = {32, wrows};
        const CUresult r0 = encode_tiled(&mw0, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, w_taps16, dims, strides, box0, sw0);
        const CUresult r1 = Cin == 96 ? encode_tiled(&mw1, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, w_taps16, dims, strides, box1, CU_TENSOR_MAP_SWIZZLE_64B)
                                      : CUDA_SUCCESS;
        if (r0 != CUDA_SUCCESS || r1 != CUDA_SUCCESS)
            return fail(MSW_ERR_ARG, "%s: weight tensor map failed (%d, %d)", who, (int)r0, (int)r1);
        if (Cin != 96) mw1 = mw0;
    }
#ifdef MSW_DEV_KNOBS
    const char *dbg_env = getenv("MSW_CONV_DBG");          // tools/convgn_ablation.py only
    const int dbg = dbg_env ? atoi(dbg_env) : 0;
#else
    const int dbg = 0;
#endif
    const ConvGnParams none = {};
    const ConvGnParams &gp = gn ? *gn : none;
    cudaStream_t st = (cudaStream_t)stream;
    if (pair) {
        if (!gn) return Cin == 128 ? conv_pair_launch_t<false, 128, 0>(ma0, ma1, mw0, mw1, y16, n, gp, max_ctas, st)
                                   : conv_pair_launch_t<false, 16, 0>(ma0, ma1, mw0, mw1, y16, n, gp, max_ctas, st);
        if (Cin == 16) return conv_pair_launch_t<true, 16, 0>(ma0, ma1, mw0, mw1, y16, n, gp, max_ctas, st);
        if (!gp.res32) return conv_pair_launch_t<true, 128, 0>(ma0, ma1, mw0, mw1, y16, n, gp, max_ctas, st);
        return gp.pool4 ? conv_pair_launch_t<true, 128, 2>(ma0, ma1, mw0, mw1, y16, n, gp, max_ctas, st)
                        : conv_pair_launch_t<true, 128, 1>(ma0, ma1, mw0, mw1, y16, n, gp, max_ctas, st);
    }
    if (!gn) return Cin == 96 ? conv_launch_t<false, 96, 0>(ma0, ma1, mw0, mw1, y16, n, dbg, gp, max_ctas, st)
                              : conv_launch_t<false, 16, 0>(ma0, ma1, mw0, mw1, y16, n, dbg, gp, max_ctas, st);
    if (Cin == 16) return conv_launch_t<true, 16, 0>(ma0, ma1, mw0, mw1, y16, n, dbg, gp, max_ctas, st);          // the stem has no residual
    if (!gp.res32) return conv_launch_t<true, 96, 0>(ma0, ma1, mw0, mw1, y16, n, dbg, gp, max_ctas, st);
    return gp.pool4 ? conv_launch_t<true, 96, 2>(ma0, ma1, mw0, mw1, y16, n, dbg, gp, max_ctas, st)
                    : conv_launch_t<true, 96, 1>(ma0, ma1, mw0, mw1, y16, n, dbg, gp, max_ctas, st);
}

extern "C" int msw_conv3x3(const void *x16, const void *w_taps16, void *y16, int64_t n, int32_t H, int32_t W,
                           int32_t Cin, int32_t C, void *stream)
{
    return conv_launch("msw_conv3x3", x16, w_taps16, y16, n, H, W, Cin, C, nullptr, 0, stream);
}

extern "C" int msw_conv3x3_gn(const void *x16, const void *w_taps16, const float *conv_bias, const float *res32,
                              const float *gamma, const float *beta, void *y16, float *y32, float *pool4, int64_t n,
                              int32_t H, int32_t W, int32_t Cin, int32_t C, int32_t G, float eps, float drop_p,
                              uint64_t seed, uint64_t call_id, const uint32_t *epoch, int64_t sample_id_base, int32_t max_ctas,
                              void *stream)
{
    using namespace msw;
    if (!conv_bias || !gamma || !beta) return fail(MSW_ERR_NULL, "msw_conv3x3_gn: NULL pointer");
    if (G != (C == 128 ? 8 : 6)) return fail(MSW_ERR_BAD_SHAPE, "msw_conv3x3_gn: needs groups of 16 channels (C=%d, G=%d)", C, G);
    if (drop_p < 0.0f || drop_p >= 1.0f) return fail(MSW_ERR_ARG, "msw_conv3x3_gn: drop_p=%f", drop_p);
    if (drop_p > 0.0f && res32) return fail(MSW_ERR_ARG, "msw_conv3x3_gn: dropout is only defined on the no-residual path");
    if (Cin != C && res32) return fail(MSW_ERR_ARG, "msw_conv3x3_gn: the residual path needs Cin = C");
    if (pool4 && (!res32 || y32)) return fail(MSW_ERR_ARG, "msw_conv3x3_gn: pool4 replaces y32 on the residual path");
    if (res32 && !pool4 && !y32) return fail(MSW_ERR_ARG, "msw_conv3x3_gn: the residual path writes y32 or pool4");
    if ((((uintptr_t)res32 | (uintptr_t)y32) & 31u) != 0)
        return fail(MSW_ERR_ALIGN, "msw_conv3x3_gn: res32 / y32 must be 32-byte aligned");
    ConvGnParams g;
    g.cbias = conv_bias; g.gamma = gamma; g.beta = beta; g.res32 = res32; g.y32 = y32; g.pool4 = pool4;
    g.eps = eps; g.drop_p = drop_p; g.drop_scale = drop_p > 0.0f ? 1.0f / (1.0f - drop_p) : 1.0f;
    g.k0 = (uint32_t)seed; g.k1 = (uint32_t)(seed >> 32);
    g.call_lo = (uint32_t)call_id; g.call_hi = (uint32_t)(call_id >> 32);
    g.epoch = epoch;
    g.sample_base = (long long)sample_id_base;
    return conv_launch("msw_conv3x3_gn", x16, w_taps16, y16, n, H, W, Cin, C, &g, max_ctas, stream);
}
