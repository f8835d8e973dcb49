// msw_cnn_fwd.cu -- the whole rollout forward of the three-convolution baseline policy (policy.CNNPolicy,
// build_model("cnn")) on 16x16 boards in ONE persistent tcgen05 kernel, as the reference runs it under fp16
// autocast (train_rl.py:222-227):
//
//   c1 = fp16(conv3x3(x16, w1) + b1)         fp32 accumulation, one rounding
//   a1 = fp16(GroupNorm_4(relu(c1)))         GroupNorm in fp32; the next convolution's input cast rounds it
//   c2 = fp16(conv3x3(a1, w2) + b2);  a2 = fp16(GroupNorm_8(relu(c2)))
//   f  = relu(fp16(conv3x3(a2, w3) + b3))    the fp16 feature map
//   policy[p] = fp16(sum_c f[p][c] * wp[c] + bp),  mine[p] = fp16(sum_c f[p][c] * wm[c] + bm)    (1x1 heads, fp32 sums)
//   pooled[c] = fp16(sum_p f[p][c] / 256)     AdaptiveAvgPool2d(1) of the fp16 features
//
// ReLU comes BEFORE GroupNorm in this network, so the conv bias is added before the ReLU (not folded into the
// GroupNorm shift as msw_conv3x3_gn does).
//
// All 27 weight taps stay resident in shared memory (119,808 B), and a board's activations never leave it: only
// the 16-channel observation (msw_pack_obs16's fp16 NHWC layout) comes in and only the logits, mine logits and
// pooled features go out.  Every convolution is msw_conv_tc.cu's scheme: per 128-pixel tile (8 image rows) nine
// shifted-descriptor taps accumulate into one TMEM accumulator, and the disable-output-lane mask switches off the
// rows whose horizontal neighbour is off the board.  A board's activation is stored with a zero halo row above and
// below (18 rows x 16 px, K-major, swizzled), so the vertical padding is those rows: the TMA box of the observation
// starts at y = -1 and the tensor map zero-fills rows -1 and 16; the epilogues write the next layer's operand into
// rows 1..16 and keep rows 0 and 17 zero.
//
// Two boards are in flight per CTA, each in its own slot of 8 warps (256 threads, thread = pixel), so that one
// board's epilogue runs under the other board's MMAs.  Slot s has two activation buffers, X (the observation, later
// conv2's output) and Y (conv1's output), and 2 x 64 TMEM columns (one accumulator per tile, reused by the three
// layers).  A slot drives its own pipeline: after each of the slot's named barriers, an elected lane of its first
// warp issues the next step, so no warp is set aside for TMA or MMA issue (16 warps leave 128 registers a thread).
// Per board:
//   conv1 MMAs (X -> TMEM, N = 32, 9 per tile) -> tfull -> epilogue: bias, round, ReLU, GroupNorm(4) -> Y -> barrier
//   conv2 MMAs (Y -> TMEM, N = 64, 18 per tile) -> tfull -> epilogue: the same with GroupNorm(8) -> X -> barrier
//   conv3 MMAs (X -> TMEM, N = 64, 36 per tile) -> tfull -> TMA of the slot's next observation into X; epilogue:
//   bias, round, ReLU, both heads, the pooled mean -> HBM
// The GroupNorm statistics span both tiles: each warp's (mean, M2) partials are merged in a fixed order after a
// barrier of the slot.
//
// Shared memory (231,472 of 232,448 B), from a 1024-byte aligned base:
//        0  W1  [9 taps][32 co][16 ch]   32-byte rows, 32-byte swizzle       9,216
//    9,216  W2  [9 taps][64 co][32 ch]   64-byte rows, 64-byte swizzle      36,864
//   46,080  W3  [9 taps][64 co][64 ch]  128-byte rows, 128-byte swizzle     73,728
//  119,808  X0  [18 rows x 16 px][16 ch (32 B rows) | 64 ch (128 B rows)]   36,864
//  156,672  Y0  [18 rows x 16 px][32 ch]  64-byte rows                      18,432
//  175,104  X1                                                              36,864
//  211,968  Y1                                                              18,432
//  230,400  GroupNorm partials [2 slots][8 warps][8 groups][mean, M2] f32    1,024
//  231,424  barriers wfull, xfull[2], tfull[2]; TMEM address                          48
// The dx = -1 tap of a tile's first row reads one pixel row before its buffer and the dx = +1 tap of the last
// row one after it; both land in the neighbouring region, in rows the mask switches off.  conv3's pooled partial
// sums ([8 warps][64] f32) borrow Y's interior rows while Y is between conv2's MMAs and the next board's conv1
// epilogue.
//
#include "../../include/msw_b200.h"
#include "msw_error.h"
#include "msw_sm100.cuh"

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace msw {

namespace cnn {
constexpr int HW_W = 16, PX = 256, PX_HALO = 18 * HW_W;         // 288 pixel rows per buffer with the halo
constexpr int CIN = 16, C1 = 32, C2 = 64, C3 = 64, G1 = 4, G2 = 8;
constexpr int THREADS = 512, SLOT_THREADS = 256, TMEM_COLS = 256;   // two slots of 8 warps
constexpr unsigned W1_TAP = C1 * 32u, W2_TAP = C2 * 64u, W3_TAP = C3 * 128u;       // bytes per weight tap
constexpr unsigned OFF_W1 = 0, OFF_W2 = OFF_W1 + 9 * W1_TAP, OFF_W3 = OFF_W2 + 9 * W2_TAP, W_BYTES = OFF_W3 + 9 * W3_TAP;
constexpr unsigned IN_BYTES = PX_HALO * 32u, X_BYTES = PX_HALO * 128u, Y_BYTES = PX_HALO * 64u;
constexpr unsigned OFF_X0 = W_BYTES, OFF_Y0 = OFF_X0 + X_BYTES, OFF_X1 = OFF_Y0 + Y_BYTES, OFF_Y1 = OFF_X1 + X_BYTES;
constexpr unsigned OFF_STAT = OFF_Y1 + Y_BYTES;
constexpr unsigned OFF_BAR = OFF_STAT + 2 * 8 * 8 * 2 * 4u;
constexpr unsigned OFF_TMEM = OFF_BAR + 5 * 8u;
constexpr unsigned SMEM_BYTES = OFF_TMEM + 8u;
static_assert(W_BYTES == 119808u, "weights");
static_assert(OFF_X0 % 1024 == 0 && OFF_Y0 % 1024 == 0 && OFF_X1 % 1024 == 0 && OFF_Y1 % 1024 == 0, "swizzle atoms");
static_assert(OFF_W2 % 512 == 0 && OFF_W3 % 1024 == 0, "swizzle atoms");
static_assert(SMEM_BYTES <= 232448, "shared memory of one CTA");
}  // namespace cnn

// Device pointers of msw_cnn_forward.  Vectors are fp32 (16-byte aligned); head weights fp16.
struct CnnParams {
    const float *b1, *g1, *be1, *b2, *g2, *be2, *b3;
    const __half *wp, *wm, *bp, *bm;
    __half *logits, *mine, *pooled;
    float eps1, eps2;
};

__device__ __forceinline__ float cnn_warp_sum(float v)           // fixed shuffle tree: deterministic
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// 16 bytes of a read-only parameter vector.  volatile: the compiler would otherwise hoist the (loop-invariant)
// bias / affine / head-weight loads out of the board loop and keep ~300 values live across it, spilling.
__device__ __forceinline__ uint4 cnn_ld16(const void *p)
{
    uint4 v;
    asm volatile("ld.global.nc.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 cnn_ldf4(const float *p)
{
    const uint4 v = cnn_ld16(p);
    return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
}

// conv3x3 of one board: for both tiles, nine taps x KS k-steps of M = 128 into d0 + 64 * tile.  `a` is the
// activation buffer (ROW bytes per pixel row, halo row first), `w` the first tap of the weights.
template <unsigned ROW, int KS>
__device__ __forceinline__ void cnn_conv_mmas(unsigned d0, unsigned a, unsigned w, unsigned wtap, unsigned idesc)
{
    // opaque per call: the 2 x 9 x KS descriptors are loop-invariant, and hoisted out of the board loop they would
    // occupy ~250 registers
    asm volatile("" : "+r"(d0), "+r"(a), "+r"(w));
#pragma unroll
    for (int t = 0; t < 2; ++t) {
        unsigned accumulate = 0u;
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
            for (int o = 0; o < 3; ++o) {
                const int dxi = o == 0 ? 1 : o == 1 ? 0 : 2;               // the unmasked centre tap first
                const int tap = dy * 3 + dxi;
                const unsigned mask = dxi == 0 ? 0x00010001u : dxi == 2 ? 0x80008000u : 0u;
                const unsigned sa = a + (unsigned)(((t * 8 + dy) * cnn::HW_W + dxi - 1) * (int)ROW);
#pragma unroll
                for (int k = 0; k < KS; ++k) {
                    umma_f16_masked(d0 + 64u * t, umma_desc<ROW>(sa) + 2u * k, umma_desc<ROW>(w + tap * wtap) + 2u * k,
                                    idesc, accumulate, mask);
                    accumulate = 1u;
                }
            }
    }
}

// 16 accumulator columns of this thread's pixel (TMEM address `taddr`, channels c0 .. c0 + 15, `bias` = &b[c0])
// -> h[0..7] = relu(fp16(acc + bias)) as half2: the conv output rounded where autocast rounds it, then the ReLU.
__device__ __forceinline__ void cnn_bias_relu16(unsigned taddr, const float *bias, uint32_t (&h)[8])
{
    uint32_t v[16];
    tmem_ld16(taddr, v);
    tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float4 bb = cnn_ldf4(bias + 4 * j);
        __half2 lo = __floats2half2_rn(__uint_as_float(v[4 * j]) + bb.x, __uint_as_float(v[4 * j + 1]) + bb.y);
        __half2 hi = __floats2half2_rn(__uint_as_float(v[4 * j + 2]) + bb.z, __uint_as_float(v[4 * j + 3]) + bb.w);
        lo = __hmax2(lo, __float2half2_rn(0.0f));
        hi = __hmax2(hi, __float2half2_rn(0.0f));
        h[2 * j] = *reinterpret_cast<const uint32_t *>(&lo);
        h[2 * j + 1] = *reinterpret_cast<const uint32_t *>(&hi);
    }
}

// The warp's (mean, M2) of one 8-channel group (h4 = 4 half2 of this thread's pixel) over its 32 pixels, written to
// st[0..1] by lane 0.  One-pass sums shifted by lane 0's first value (no cancellation in S2 - S1^2 / n).
__device__ __forceinline__ void cnn_group_partial(const uint32_t *h4, float *st, int lane)
{
    const float shift = __shfl_sync(0xffffffffu, __low2float(*reinterpret_cast<const __half2 *>(&h4[0])), 0);
    float s1 = 0.0f, s2 = 0.0f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&h4[k]));
        const float d0 = f.x - shift, d1 = f.y - shift;
        s1 += d0 + d1;
        s2 = fmaf(d0, d0, fmaf(d1, d1, s2));
    }
    s1 = cnn_warp_sum(s1);
    s2 = cnn_warp_sum(s2);
    if (lane == 0) {
        st[0] = shift + s1 * (1.0f / 256.0f);
        st[1] = s2 - s1 * s1 * (1.0f / 256.0f);
    }
}

// The board's GroupNorm of group g from the eight warps' (mean, M2) partials, merged in a fixed order (Chan et
// al.; every thread merges the same numbers the same way): returns (mean, rstd) with the biased variance.
__device__ __forceinline__ float2 cnn_group_stats(const float *stat, int g, float eps)
{
    float na = 0.0f, mg = 0.0f, m2 = 0.0f;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        const float2 pw = *reinterpret_cast<const float2 *>(stat + (w * 8 + g) * 2);
        const float nn = na + 256.0f, delta = pw.x - mg, r = 256.0f / nn;
        mg = fmaf(delta, r, mg);
        m2 += pw.y + delta * delta * (na * r);
        na = nn;
    }
    return make_float2(mg, rsqrtf(m2 * (1.0f / 2048.0f) + eps));
}

// Normalise 8 channels (group g = chunk) of this thread's pixel: fp16(relu-output * a + b), a = gamma * rstd,
// b = beta - mean * a, packed as one 16-byte chunk.
__device__ __forceinline__ uint4 cnn_norm8(const uint32_t *h, const float *gamma, const float *beta, float2 ms)
{
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float4 gg = cnn_ldf4(gamma + 4 * j), bb = cnn_ldf4(beta + 4 * j);
        const float gv[4] = {gg.x, gg.y, gg.z, gg.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
        for (int k = 0; k < 4; k += 2) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&h[(4 * j + k) >> 1]));
            const float a0 = gv[k] * ms.y, a1 = gv[k + 1] * ms.y;
            const __half2 hh = __floats2half2_rn(fmaf(f.x, a0, fmaf(-ms.x, a0, bv[k])), fmaf(f.y, a1, fmaf(-ms.x, a1, bv[k + 1])));
            o[(4 * j + k) >> 1] = *reinterpret_cast<const uint32_t *>(&hh);
        }
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
}

__device__ __forceinline__ void cnn_st_shared16(unsigned addr, uint4 v)
{
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" :: "r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__global__ void __launch_bounds__(cnn::THREADS, 1)
cnn_fwd_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w1,
               const __grid_constant__ CUtensorMap map_w2, const __grid_constant__ CUtensorMap map_w3,
               const __grid_constant__ CnnParams prm, long long boards)
{
    using namespace cnn;
    extern __shared__ __align__(1024) unsigned char smem_cnn[];
    const unsigned base = smem_u32(smem_cnn);
    if (base & 1023u) {                  // the layout has no room to realign; uniform over the grid
        if (threadIdx.x == 0 && blockIdx.x == 0) printf("cnn_fwd_kernel: dynamic shared memory is not 1024-byte aligned\n");
        return;
    }
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // slot s = warps 8s .. 8s + 7; warp 8s + 4t + q owns pixels 128t + 32q .. +31 (TMEM lanes 32q .. +31 of tile t)
    const unsigned s = (unsigned)(warp >> 3);
    const int wi = warp & 7, q = warp & 3, t = (warp >> 2) & 1, p = t * 128 + q * 32 + lane;
    const bool leader = wi == 0;                                       // its elected lane issues the slot's TMA and MMAs
    const unsigned bars = base + OFF_BAR, wfull = bars, xfull = bars + 8u * (1 + s), tfull = bars + 8u * (3 + s);
    const unsigned xa = base + (s ? OFF_X1 : OFF_X0), ya = base + (s ? OFF_Y1 : OFF_Y0);
    volatile uint32_t *s_tmem = reinterpret_cast<volatile uint32_t *>(smem_cnn + OFF_TMEM);
    auto slot_sync = [&]() {                                           // the slot's 256 threads (named barrier 1 + s)
        if (s == 0) asm volatile("bar.sync 1, %0;" :: "n"(SLOT_THREADS) : "memory");
        else asm volatile("bar.sync 2, %0;" :: "n"(SLOT_THREADS) : "memory");
    };
    auto board_of = [&](unsigned i) { return blockIdx.x + (long long)(2 * i + s) * gridDim.x; };

    if (tid == 0) {
        mbar_init(wfull, 1);
        for (unsigned k = 1; k < 5; ++k) mbar_init(bars + 8u * k, 1);    // xfull[2], tfull[2]
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(base + OFF_TMEM, TMEM_COLS);
    // conv1's output buffers are zeroed once: nothing writes their halo rows afterwards
    for (unsigned k = tid; k < 2 * Y_BYTES / 16; k += THREADS) {
        const unsigned y = k >= Y_BYTES / 16, off = (k - y * (Y_BYTES / 16)) * 16u;
        cnn_st_shared16(base + (y ? OFF_Y1 : OFF_Y0) + off, make_uint4(0u, 0u, 0u, 0u));
    }
    fence_proxy_async();
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const unsigned tmem = *s_tmem;
    const unsigned d0 = tmem + s * 128u;                               // the slot's two accumulators (64 columns each)
    const unsigned tl = tmem + ((unsigned)(q * 32) << 16) + s * 128u + 64u * t;   // this warp's rows of its tile
    float *stat = reinterpret_cast<float *>(smem_cnn + OFF_STAT) + s * 128;        // [8 warps][8 groups][mean, M2]
    float *wstat = stat + wi * 16;
    float *pool_part = reinterpret_cast<float *>(smem_cnn + (s ? OFF_Y1 : OFF_Y0) + 16 * 64);   // [8 warps][64], Y's interior
    // idesc: D = F32, A = B = F16, K-major, M = 128, N = 32 / 64
    constexpr unsigned id32 = (1u << 4) | ((unsigned)(C1 >> 3) << 17) | ((128u >> 4) << 24);
    constexpr unsigned id64 = (1u << 4) | ((unsigned)(C2 >> 3) << 17) | ((128u >> 4) << 24);

    if (leader && elect_one()) {
        if (s == 0) {                                                  // the 27 weight taps, once per CTA
            mbar_expect_tx(wfull, W_BYTES);
            for (int k = 0; k < 9; ++k) {
                tma_load_2d(base + OFF_W1 + k * W1_TAP, &map_w1, 0, k * C1, wfull);
                tma_load_2d(base + OFF_W2 + k * W2_TAP, &map_w2, 0, k * C2, wfull);
                tma_load_2d(base + OFF_W3 + k * W3_TAP, &map_w3, 0, k * C3, wfull);
            }
        }
        if (board_of(0) < boards) {
            mbar_expect_tx(xfull, IN_BYTES);
            tma_load_4d(xa, &map_x, 0, 0, -1, (int)board_of(0), xfull);  // rows -1 and 16 zero-filled
        }
    }
    // tfull completes three times per board (conv1, conv2, conv3): completion 3i + l has parity (3i + l) & 1
    for (unsigned i = 0;; ++i) {
        const long long board = board_of(i);
        if (board >= boards) break;
        // ---- conv1 (X -> TMEM).  TMEM is free: every thread read the previous board's conv3 accumulator before the
        //      barrier that ended the last iteration.
        if (leader) {
            if (elect_one()) {
                if (i == 0) mbar_wait(wfull, 0);
                mbar_wait(xfull, i & 1u);
                tcgen05_fence_after();
                cnn_conv_mmas<32u, 1>(d0, xa, base + OFF_W1, W1_TAP, id32);
                umma_commit(tfull);
            }
            __syncwarp();
        }
        // ---- conv1 epilogue: bias, fp16, ReLU, GroupNorm(4) -> Y (64-byte rows, 64-byte swizzle).  The accumulator
        //      stays in TMEM until the next MMA, so it is read twice (statistics, then normalise) instead of being held
        //      in registers across the barrier.
        mbar_wait(tfull, (3 * i) & 1u);
        tcgen05_fence_after();
#pragma unroll
        for (int c = 0; c < C1 / 16; ++c) {
            uint32_t h[8];
            cnn_bias_relu16(tl + 16 * c, prm.b1 + 16 * c, h);
            cnn_group_partial(h, wstat + 4 * c, lane);
            cnn_group_partial(h + 4, wstat + 4 * c + 2, lane);
        }
        slot_sync();
        const int row = p + HW_W;                                      // pixel row in a halo'd buffer
#pragma unroll
        for (int c = 0; c < C1 / 16; ++c) {
            uint32_t h[8];
            cnn_bias_relu16(tl + 16 * c, prm.b1 + 16 * c, h);
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const unsigned g = 2 * c + u;
                const uint4 o = cnn_norm8(h + 4 * u, prm.g1 + 8 * g, prm.be1 + 8 * g, cnn_group_stats(stat, g, prm.eps1));
                cnn_st_shared16(ya + row * 64u + ((g ^ ((row >> 1) & 3u)) << 4), o);
            }
        }
        fence_proxy_async();                                           // Y -> the tensor cores
        tcgen05_fence_before();
        slot_sync();
        // ---- conv2 (Y -> TMEM)
        if (leader) {
            if (elect_one()) {
                tcgen05_fence_after();
                cnn_conv_mmas<64u, 2>(d0, ya, base + OFF_W2, W2_TAP, id64);
                umma_commit(tfull);
            }
            __syncwarp();
        }
        // ---- conv2 epilogue: the same with GroupNorm(8) -> X (128-byte rows, 128-byte swizzle); X's halo rows are
        //      zeroed again (the observation's TMA load wrote over the top one)
        mbar_wait(tfull, (3 * i + 1) & 1u);
        tcgen05_fence_after();
#pragma unroll
        for (int c = 0; c < C2 / 16; ++c) {
            uint32_t h[8];
            cnn_bias_relu16(tl + 16 * c, prm.b2 + 16 * c, h);
            cnn_group_partial(h, wstat + 4 * c, lane);
            cnn_group_partial(h + 4, wstat + 4 * c + 2, lane);
        }
        slot_sync();
#pragma unroll
        for (int c = 0; c < C2 / 16; ++c) {
            uint32_t h[8];
            cnn_bias_relu16(tl + 16 * c, prm.b2 + 16 * c, h);
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const unsigned g = 2 * c + u;
                const uint4 o = cnn_norm8(h + 4 * u, prm.g2 + 8 * g, prm.be2 + 8 * g, cnn_group_stats(stat, g, prm.eps2));
                cnn_st_shared16(xa + row * 128u + ((g ^ (row & 7u)) << 4), o);
            }
        }
        cnn_st_shared16(xa + (p < 128 ? p * 16u : 17u * 16u * 128u + (p - 128) * 16u), make_uint4(0u, 0u, 0u, 0u));
        fence_proxy_async();
        tcgen05_fence_before();
        slot_sync();
        // ---- conv3 (X -> TMEM)
        if (leader) {
            if (elect_one()) {
                tcgen05_fence_after();
                cnn_conv_mmas<128u, 4>(d0, xa, base + OFF_W3, W3_TAP, id64);
                umma_commit(tfull);
            }
            __syncwarp();
        }
        // ---- conv3 epilogue: bias, fp16, ReLU -> both 1x1 heads (fp32 sums over the 64 channels), pooled mean
        mbar_wait(tfull, (3 * i + 2) & 1u);
        tcgen05_fence_after();
        if (leader && board_of(i + 1) < boards) {                      // conv3 has read X: the next observation may land
            if (elect_one()) {
                mbar_expect_tx(xfull, IN_BYTES);
                tma_load_4d(xa, &map_x, 0, 0, -1, (int)board_of(i + 1), xfull);
            }
            __syncwarp();
        }
        float pol = 0.0f, mn = 0.0f;
#pragma unroll
        for (int c = 0; c < C3 / 16; ++c) {
            uint32_t f[8];                                             // the fp16 features, channels 16c + 2j, + 1
            cnn_bias_relu16(tl + 16 * c, prm.b3 + 16 * c, f);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const uint4 wpv = cnn_ld16(prm.wp + 16 * c + 8 * j), wmv = cnn_ld16(prm.wm + 16 * c + 8 * j);
                const uint32_t wpw[4] = {wpv.x, wpv.y, wpv.z, wpv.w}, wmw[4] = {wmv.x, wmv.y, wmv.z, wmv.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float2 x = __half22float2(*reinterpret_cast<const __half2 *>(&f[4 * j + k]));
                    const float2 ap = __half22float2(*reinterpret_cast<const __half2 *>(&wpw[k]));
                    const float2 am = __half22float2(*reinterpret_cast<const __half2 *>(&wmw[k]));
                    pol = fmaf(x.y, ap.y, fmaf(x.x, ap.x, pol));
                    mn = fmaf(x.y, am.y, fmaf(x.x, am.x, mn));
                }
            }
            // the warp's sums of these 16 channels over its 32 pixels by recursive halving (a fixed butterfly:
            // deterministic): each step a lane keeps half of its channels and adds the partner's copy of them.  The
            // first step adds two fp16 values, exact in fp32; lanes 2m and 2m + 1 end with channel 16c + m.
            float a[8];
            {
                const bool up = lane & 16;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t keep = up ? f[4 + j] : f[j], send = up ? f[j] : f[4 + j];
                    const uint32_t got = __shfl_xor_sync(0xffffffffu, send, 16);
                    const float2 x = __half22float2(*reinterpret_cast<const __half2 *>(&keep));
                    const float2 y = __half22float2(*reinterpret_cast<const __half2 *>(&got));
                    a[2 * j] = x.x + y.x;
                    a[2 * j + 1] = x.y + y.y;
                }
            }
#pragma unroll
            for (int m = 8; m >= 2; m >>= 1) {                         // 8, 4, 2 channels -> half of them
                const bool up = lane & m;
#pragma unroll
                for (int j = 0; j < m / 2; ++j) {
                    const float keep = up ? a[m / 2 + j] : a[j], send = up ? a[j] : a[m / 2 + j];
                    a[j] = keep + __shfl_xor_sync(0xffffffffu, send, m);
                }
            }
            a[0] += __shfl_xor_sync(0xffffffffu, a[0], 1);
            if ((lane & 1) == 0) pool_part[wi * 64 + 16 * c + (lane >> 1)] = a[0];
        }
        tcgen05_fence_before();
        slot_sync();                       // TMEM has been read (the next conv1 may overwrite it); pool_part is complete
        const long long px = board * PX + p;
        prm.logits[px] = __float2half_rn(pol + __half2float(*prm.bp));
        prm.mine[px] = __float2half_rn(mn + __half2float(*prm.bm));
        if (p < C3) {
            float sum = 0.0f;
#pragma unroll
            for (int w = 0; w < 8; ++w) sum += pool_part[w * 64 + p];
            prm.pooled[board * C3 + p] = __float2half_rn(sum * (1.0f / 256.0f));
        }
    }

    tcgen05_fence_before();
    __syncthreads();
    if (warp == 0) {
        tcgen05_fence_after();
        tmem_dealloc(*s_tmem, TMEM_COLS);                              // re-read: not worth a register across the loop
    }
}

}  // namespace msw

extern "C" int msw_cnn_forward(const void *x16, const void *w1_taps16, const float *b1, const float *gamma1,
                               const float *beta1, const void *w2_taps16, const float *b2, const float *gamma2,
                               const float *beta2, const void *w3_taps16, const float *b3, const void *wp16,
                               const void *bp16, const void *wm16, const void *bm16, void *logits16, void *mine16,
                               void *pooled16, int64_t n, int32_t H, int32_t W, int32_t Cin, int32_t C1, int32_t G1,
                               int32_t C2, int32_t G2, int32_t C3, float eps1, float eps2, void *stream)
{
    using namespace msw;
    const void *ptrs[18] = {x16, w1_taps16, b1, gamma1, beta1, w2_taps16, b2, gamma2, beta2, w3_taps16, b3, wp16, bp16, wm16,
                            bm16, logits16, mine16, pooled16};
    for (const void *q : ptrs)
        if (!q) return fail(MSW_ERR_NULL, "msw_cnn_forward: NULL pointer");
    if (H != 16 || W != 16 || Cin != cnn::CIN || C1 != cnn::C1 || G1 != cnn::G1 || C2 != cnn::C2 || G2 != cnn::G2 || C3 != cnn::C3)
        return fail(MSW_ERR_BAD_SHAPE,
                    "msw_cnn_forward: only 16x16 boards, 16 packed input channels and widths 32 / 64 / 64 with 4 / 8 groups "
                    "(got %dx%d, Cin %d, widths %d / %d / %d, groups %d / %d)", H, W, Cin, C1, C2, C3, G1, G2);
    if (n < 0 || n > 0x3fffffffLL) return fail(MSW_ERR_BAD_SHAPE, "msw_cnn_forward: n=%lld", (long long)n);
    for (int k = 0; k < 15; ++k)
        if (k != 12 && k != 14 && ((uintptr_t)ptrs[k] & 15u) != 0)
            return fail(MSW_ERR_ALIGN, "msw_cnn_forward: inputs, weights and fp32 vectors must be 16-byte aligned");
    if ((((uintptr_t)bp16 | (uintptr_t)bm16 | (uintptr_t)logits16 | (uintptr_t)mine16 | (uintptr_t)pooled16) & 1u) != 0)
        return fail(MSW_ERR_ALIGN, "msw_cnn_forward: fp16 outputs and head biases must be 2-byte aligned");
    if (n == 0) return MSW_OK;
    if (!tensor_map_encoder_available()) return fail(MSW_ERR_ARG, "msw_cnn_forward: cuTensorMapEncodeTiled is not available");
    CUtensorMap mx, mw1, mw2, mw3;
    {
        // observation [n][16][16][16] fp16 NHWC, innermost first; one board per box with rows -1 .. 16
        const cuuint64_t dims[4] = {16, 16, 16, (cuuint64_t)n};
        const cuuint64_t strides[3] = {32, 32 * 16, 32 * 256};
        const cuuint32_t box[4] = {16, 16, 18, 1};
        const CUresult r = encode_tiled(&mx, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, x16, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_32B);
        if (r != CUDA_SUCCESS) return fail(MSW_ERR_ARG, "msw_cnn_forward: input tensor map failed (%d)", (int)r);
    }
    {
        // weights [9 taps * Cout][Cin] fp16, one tap per box
        const void *w[3] = {w1_taps16, w2_taps16, w3_taps16};
        const cuuint32_t cin[3] = {16, 32, 64}, cout[3] = {32, 64, 64};
        const CUtensorMapSwizzle sw[3] = {CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_SWIZZLE_128B};
        CUtensorMap *m[3] = {&mw1, &mw2, &mw3};
        for (int l = 0; l < 3; ++l) {
            const cuuint64_t dims[2] = {cin[l], (cuuint64_t)9 * cout[l]};
            const cuuint64_t strides[1] = {(cuuint64_t)cin[l] * 2};
            const cuuint32_t box[2] = {cin[l], cout[l]};
            const CUresult r = encode_tiled(m[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, w[l], dims, strides, box, sw[l]);
            if (r != CUDA_SUCCESS) return fail(MSW_ERR_ARG, "msw_cnn_forward: weight tensor map %d failed (%d)", l + 1, (int)r);
        }
    }
    CnnParams prm;
    prm.b1 = b1; prm.g1 = gamma1; prm.be1 = beta1; prm.b2 = b2; prm.g2 = gamma2; prm.be2 = beta2; prm.b3 = b3;
    prm.wp = (const __half *)wp16; prm.wm = (const __half *)wm16; prm.bp = (const __half *)bp16; prm.bm = (const __half *)bm16;
    prm.logits = (__half *)logits16; prm.mine = (__half *)mine16; prm.pooled = (__half *)pooled16;
    prm.eps1 = eps1; prm.eps2 = eps2;
    MSW_SET_MAX_SMEM(cnn_fwd_kernel, cnn::SMEM_BYTES);
    const long long sms = sm_count();
    const long long grid = n < sms ? n : sms;                         // persistent: two boards in flight per CTA
    cnn_fwd_kernel<<<(unsigned)grid, cnn::THREADS, cnn::SMEM_BYTES, (cudaStream_t)stream>>>(mx, mw1, mw2, mw3, prm, (long long)n);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}
