// msw_conv_tc.cu -- 3x3 "same" convolution of the policy trunk on 16x16 boards (fp16 NHWC in, fp32 accumulate, fp16
// NHWC out) on the 5th-generation tensor cores, plain (GN = false: no bias, it is folded into msw_gn_act) or with
// GroupNorm / ReLU / Dropout2d / residual add (and the value head's average pool) fused into the epilogue (GN = true).
//   * 96 -> 96 channels and the stem's 16 -> 96: conv3x3_tc_kernel, one board per CTA;
//   * 128 -> 128 channels and the stem's 16 -> 128: conv3x3_pair_kernel below, one board per CTA pair.
// The shifted-descriptor / edge-mask scheme of the nine taps, the GroupNorm statistics, the pooled-sum butterfly and
// the P8 order of the fp32 residual stream are in msw_conv.cuh; the mbarrier / TMA / tcgen05 wrappers in msw_sm100.cuh.
//
// conv3x3_tc_kernel: all nine [96 x 96] weight taps stay resident in shared memory (162 KB, loaded once per persistent
// CTA); the activation streams through a 2-stage ring of [10 rows x 16 px x 96 ch] blocks (a single 4-D TMA box; rows
// above / below the board are zero-filled by the tensor map).  K = 96 = one 64-channel block (128-byte swizzle) + one
// 32-channel block (64-byte swizzle).  Roles: warp 0 TMA producer, warp 1 MMA issuer (54 tcgen05.mma of 128 x 96 x 16
// per tile into a ring of four 96-column accumulators), warp 2 TMEM allocation, warps 4-15 epilogue (thread = pixel,
// each warpgroup a third of the channels).
#include "../../include/msw_b200.h"
#include "msw_common.cuh"
#include "msw_conv.cuh"
#include "msw_error.h"
#include "msw_sm100.cuh"

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

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

// What the fused GroupNorm epilogue needs (GN = true); same meaning as msw_gn_act's arguments.  The fp32 residual
// stream (res32 in, y32 out) is private to this kernel family, so it is kept in the P8 order of msw_conv.cuh.
struct ConvGnParams {
    const float *cbias, *gamma, *beta;   // [C]
    const float *res32;                  // nullable, P8 order
    float *y32;                          // nullable, P8 order
    float *pool4;                        // nullable [n][4][96]: per row-quarter sums of the fp32 output (value head's avg pool)
    float eps, drop_p, drop_scale;
    uint32_t k0, k1, call_lo, call_hi;
    const uint32_t *epoch;               // nullable
    long long sample_base;               // global index of board 0 (Dropout2d stream is keyed by the global board)
};

// GN = false: out = conv(x) (fp16).  GN = true: out = relu(GroupNorm(conv(x) + bias) [+ res]) [* Dropout2d], the
// whole inter-convolution step of msw_gn_act fused into the epilogue (6 groups of 16 channels; statistics over
// the board = the CTA's two consecutive tiles, whose fp16-rounded conv outputs wait in registers).
// EPI (GN only): 0 = no residual (Dropout2d allowed, y32 optional), 1 = residual in, y32 out, 2 = residual in, pooled
// sums out (the last block: nothing reads its residual stream but the value head's average pool).
template <bool GN, int CIN, int EPI>
__global__ void __launch_bounds__(cv::THREADS, 1)
conv3x3_tc_kernel(const __grid_constant__ CUtensorMap map_a0, const __grid_constant__ CUtensorMap map_a1,
                  const __grid_constant__ CUtensorMap map_w0, const __grid_constant__ CUtensorMap map_w1,
                  __half *__restrict__ out, long long boards, const __grid_constant__ ConvGnParams gp)
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
            conv3x3_mmas<K::ROW0, K::KS0, K::ROW1, K::KS1, false>(d, a0, a1, base + OFF_W0, base + OFF_W1, W0_TAP, W1_TAP, idesc);
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
            uint32_t lo[16], hi[16];
            const unsigned taddr = tmem + ((unsigned)(q * 32) << 16) + acc * C + third * 32;
            tmem_ld16(taddr, lo);
            tmem_ld16(taddr + 16, hi);
            tmem_wait_ld();
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty(acc));       // the accumulator is in registers: release it
            store_half32(out + (board * 256 + (it & 1u) * 128 + q * 32 + lane) * (long long)C + third * 32, lo, hi);
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
                dropout2d_draw(gp.k0, gp.k1, gp.sample_base + board, (uint32_t)(te >> 3), gp.call_lo, gp.call_hi, gp.epoch, w);
                if (dropout2d_u16(w, te & 7) < thresh) sc = 0.0f;
            }
            uint32_t h[2][16];                       // fp16-rounded conv output of both tiles (the reference's rounding point)
            GnSums sums = {};
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const unsigned it = 2u * bi + half, acc = it % ACC, aph = (it / ACC) & 1u;
                if (EPI != 0)     // the 16 KB of residual stream this warpgroup will read for this tile: one line per thread on its way to L2
                    asm volatile("prefetch.global.L2 [%0];" :: "l"(gp.res32 + p8_offset<3>(board, half, third, 0, 0) + (q * 32 + lane) * 32));
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
                gn_accumulate32(lo, hi, cb2, half == 0, h[half], sums);
            }
            // the warp's (mean, M2) over its 1,024 values per group; the board's statistics are merged from the four
            // row-owning warps of a channel third in a fixed order
            const float s1a = warp_sum(sums.s1[0]), s2a = warp_sum(sums.s2[0]), s1b = warp_sum(sums.s1[1]), s2b = warp_sum(sums.s2[1]);
            if (lane == 0) {
                const float2 st0 = mean_m2<1024>(sums.shift[0], s1a, s2a), st1 = mean_m2<1024>(sums.shift[1], s1b, s2b);
                float *dst = s_part + (par * 12 + we) * 4;
                dst[0] = st0.x; dst[1] = st0.y;
                dst[2] = st1.x; dst[3] = st1.y;
            }
            asm volatile("bar.sync 1, 384;" ::: "memory");
            if (te < C) {
                // one thread per channel folds statistics, affine, conv bias and the Dropout2d scale into y = a*x + b
                const int c = te, gsel = (c >> 4) & 1, w4 = (c >> 5) * 4;
                float na = 0.0f, mg = 0.0f, m2 = 0.0f;
#pragma unroll
                for (int qq = 0; qq < 4; ++qq) {
                    const float *src = s_part + (par * 12 + w4 + qq) * 4 + 2 * gsel;
                    chan_step(na, mg, m2, 1024.0f, src[0], src[1]);
                }
                const float2 ab = gn_fold<4096>(mg, m2, gp.eps, gp.gamma[c], gp.beta[c], s_cb[c], sc);
                s_ab[(par * 2 + 0) * C + c] = ab.x;
                s_ab[(par * 2 + 1) * C + c] = ab.y;
            }
            asm volatile("bar.sync 1, 384;" ::: "memory");
            // ---- normalise, (+ residual), ReLU, store: chunk by chunk (8 channels), both tiles per chunk
            const float4 *a4 = reinterpret_cast<const float4 *>(s_ab + (par * 2 + 0) * C + cbase);
            const float4 *b4 = reinterpret_cast<const float4 *>(s_ab + (par * 2 + 1) * C + cbase);
            const int pp = q * 32 + lane;
            uint32_t rnext[8];                       // residual values of the next (chunk, tile): loaded one step ahead
            if (EPI != 0) ld256(gp.res32 + p8_offset<3>(board, 0, third, 0, pp), rnext);
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
                        if (half == 0) ld256(gp.res32 + p8_offset<3>(board, 1, third, c0 >> 3, pp), rnext);
                        else if (c0 < 24) ld256(gp.res32 + p8_offset<3>(board, 0, third, (c0 >> 3) + 1, pp), rnext);
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
                    if (EPI != 2 && gp.y32) st256(gp.y32 + p8_offset<3>(board, half, third, c0 >> 3, pp), o);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const __half2 hh = __floats2half2_rn(__uint_as_float(o[2 * k]), __uint_as_float(o[2 * k + 1]));
                        h[half][(c0 >> 1) + k] = *reinterpret_cast<const uint32_t *>(&hh);     // reuse the slot for the output
                    }
                }
                if (EPI == 2) {                      // the warp's sum of these 8 channels over its 32 pixels
                    int ch;
                    const float sum = pool8_butterfly(ps, lane, ch);
                    if ((lane & 3) == 0) gp.pool4[(board * 4 + q) * C + cbase + c0 + ch] = sum;
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
                    st256(out + px * C + cbase + c0, packed);
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
// 128 pixels x all 128 output channels.  The taps are msw_conv.cuh's conv3x3_mmas in its pair form.  K = 128 = two
// 64-channel blocks (128-byte rows, 128-byte swizzle; both through the same tensor map); the stem (CIN = 16) is as
// above.
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
constexpr int C = 128, HALF = 64, TILE_PX = 128, PX_IN = 160;
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
            conv3x3_mmas<K::ROW0, K::KS0, K::ROW1, K::KS1, true>(d, a0, a1, base + K::OFF_W0, base + K::OFF_W1, W0_TAP, W1_TAP, idesc);
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
            store_half32(out + (board * 256 + rank * 128 + pp) * (long long)C + cbase, lo, hi);
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
                dropout2d_draw(gp.k0, gp.k1, gp.sample_base + board, (uint32_t)(te >> 3), gp.call_lo, gp.call_hi, gp.epoch, w);
                if (dropout2d_u16(w, te & 7) < thresh) sc = 0.0f;
            }
            if (EPI != 0)     // the 16 KB of residual stream this warpgroup reads for this tile: one line per thread
                asm volatile("prefetch.global.L2 [%0];" :: "l"(gp.res32 + p8_offset<4>(board, (int)rank, wg, 0, 0) + pp * 32));
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
            GnSums sums = {};
            gn_accumulate32(lo, hi, cb2, true, h, sums);
            // the warp's (mean, M2) of its 512 values per group, into both CTAs' exchange areas
            const float s1a = warp_sum(sums.s1[0]), s2a = warp_sum(sums.s2[0]), s1b = warp_sum(sums.s1[1]), s2b = warp_sum(sums.s2[1]);
            if (lane == 0) {
                const float2 st0 = mean_m2<512>(sums.shift[0], s1a, s2a), st1 = mean_m2<512>(sums.shift[1], s1b, s2b);
                const float4 st = make_float4(st0.x, st0.y, st1.x, st1.y);
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
                        chan_step(na, mg, m2, 512.0f, src[0], src[1]);
                    }
                const float2 ab = gn_fold<4096>(mg, m2, gp.eps, gp.gamma[c], gp.beta[c], s_cb[c], sc);
                s_ab[c] = ab.x;
                s_ab[C + c] = ab.y;
            }
            asm volatile("bar.sync 1, 512;" ::: "memory");
            // ---- normalise, (+ residual), ReLU, store: 8 channels at a time
            const float4 *a4 = reinterpret_cast<const float4 *>(s_ab + cbase);
            const float4 *b4 = reinterpret_cast<const float4 *>(s_ab + C + cbase);
            uint32_t rnext[8];
            if (EPI != 0) ld256(gp.res32 + p8_offset<4>(board, (int)rank, wg, 0, pp), rnext);
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 8) {
                const float4 aa0 = a4[c0 >> 2], aa1 = a4[(c0 >> 2) + 1], bb0 = b4[c0 >> 2], bb1 = b4[(c0 >> 2) + 1];
                const float av[8] = {aa0.x, aa0.y, aa0.z, aa0.w, aa1.x, aa1.y, aa1.z, aa1.w};
                const float bv[8] = {bb0.x, bb0.y, bb0.z, bb0.w, bb1.x, bb1.y, bb1.z, bb1.w};
                uint32_t rr[8];
                if (EPI != 0) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) rr[k] = rnext[k];
                    if (c0 < 24) ld256(gp.res32 + p8_offset<4>(board, (int)rank, wg, (c0 >> 3) + 1, pp), rnext);
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
                if (EPI != 2 && gp.y32) st256(gp.y32 + p8_offset<4>(board, (int)rank, wg, c0 >> 3, pp), o);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const __half2 hh = __floats2half2_rn(__uint_as_float(o[2 * k]), __uint_as_float(o[2 * k + 1]));
                    h[(c0 >> 1) + k] = *reinterpret_cast<const uint32_t *>(&hh);
                }
                if (EPI == 2) {                      // the warp's sum of these 8 channels over its 32 pixels
                    float ps[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) ps[k] = __uint_as_float(o[k]);
                    int ch;
                    const float sum = pool8_butterfly(ps, lane, ch);
                    if ((lane & 3) == 0) gp.pool4[(board * 8 + rank * 4 + q) * C + cbase + c0 + ch] = sum;
                }
            }
            __half *dst = out + (board * 256 + rank * 128 + pp) * (long long)C + cbase;
#pragma unroll
            for (int c0 = 0; c0 < 32; c0 += 16) {
                uint32_t packed[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) packed[k] = h[(c0 >> 1) + k];
                st256(dst + c0, packed);
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

// Launch of either family with the kernel for <GN, stem, EPI>: conv3x3_tc_kernel (C = 96, one CTA per board) or, for
// `pair`, conv3x3_pair_kernel (C = 128) in clusters of 2, one board per cluster at a time, at most one cluster per two
// SMs.
template <bool GN, bool STEM, int EPI>
static int conv_launch_t(bool pair, const CUtensorMap &ma0, const CUtensorMap &ma1, const CUtensorMap &mw0, const CUtensorMap &mw1,
                         void *y16, int64_t n, const msw::ConvGnParams &gp, cudaStream_t stream)
{
    using namespace msw;
    constexpr int CIN96 = STEM ? 16 : 96, CIN128 = STEM ? 16 : 128;
    const unsigned smem = pair ? cvp::Cfg<CIN128>::SMEM_BYTES : cv::Cfg<CIN96>::SMEM_BYTES;
    if (pair) MSW_SET_MAX_SMEM((conv3x3_pair_kernel<GN, CIN128, EPI>), smem);
    else MSW_SET_MAX_SMEM((conv3x3_tc_kernel<GN, CIN96, EPI>), smem);
    const int sms = sm_count();
    // persistent: whole boards per CTA (per CTA pair)
    const long long units_max = pair ? (sms / 2 > 0 ? sms / 2 : 1) : sms;
    const long long units = n < units_max ? n : units_max;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(pair ? 2 * units : units), 1, 1);
    cfg.blockDim = dim3(pair ? cvp::THREADS : cv::THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pair ? 1 : 0;
    MSW_CUDA_TRY(cudaLaunchKernelEx(&cfg, pair ? conv3x3_pair_kernel<GN, CIN128, EPI> : conv3x3_tc_kernel<GN, CIN96, EPI>, ma0, ma1,
                                    mw0, mw1, (__half *)y16, (long long)n, gp));
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

// Shared host side of msw_conv3x3 / msw_conv3x3_gn: argument checks, the four tensor maps, the launch.
// C = 96 (Cin 96 or 16): conv3x3_tc_kernel, one CTA per board; C = 128 (Cin 128 or 16): conv3x3_pair_kernel.
static int conv_launch(const char *who, const void *x16, const void *w_taps16, void *y16, int64_t n, int32_t H, int32_t W,
                       int32_t Cin, int32_t C, const msw::ConvGnParams *gn, void *stream)
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
    const ConvGnParams none = {};
    const ConvGnParams &gp = gn ? *gn : none;
    const bool stem = Cin == 16;
    cudaStream_t st = (cudaStream_t)stream;
    if (!gn) return stem ? conv_launch_t<false, true, 0>(pair, ma0, ma1, mw0, mw1, y16, n, gp, st)
                         : conv_launch_t<false, false, 0>(pair, ma0, ma1, mw0, mw1, y16, n, gp, st);
    if (stem) return conv_launch_t<true, true, 0>(pair, ma0, ma1, mw0, mw1, y16, n, gp, st);      // the stem has no residual
    if (!gp.res32) return conv_launch_t<true, false, 0>(pair, ma0, ma1, mw0, mw1, y16, n, gp, st);
    return gp.pool4 ? conv_launch_t<true, false, 2>(pair, ma0, ma1, mw0, mw1, y16, n, gp, st)
                    : conv_launch_t<true, false, 1>(pair, ma0, ma1, mw0, mw1, y16, n, gp, st);
}

extern "C" int msw_conv3x3(const void *x16, const void *w_taps16, void *y16, int64_t n, int32_t H, int32_t W,
                           int32_t Cin, int32_t C, void *stream)
{
    return conv_launch("msw_conv3x3", x16, w_taps16, y16, n, H, W, Cin, C, nullptr, stream);
}

extern "C" int msw_conv3x3_gn(const void *x16, const void *w_taps16, const float *conv_bias, const float *res32,
                              const float *gamma, const float *beta, void *y16, float *y32, float *pool4, int64_t n,
                              int32_t H, int32_t W, int32_t Cin, int32_t C, int32_t G, float eps, float drop_p,
                              uint64_t seed, uint64_t call_id, const uint32_t *epoch, int64_t sample_id_base, void *stream)
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
    return conv_launch("msw_conv3x3_gn", x16, w_taps16, y16, n, H, W, Cin, C, &g, stream);
}
