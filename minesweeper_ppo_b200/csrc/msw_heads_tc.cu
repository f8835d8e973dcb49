// msw_heads_tc.cu -- the per-cell heads of msw_heads.cu on the 5th-generation tensor cores.
//
// Same operation and rounding points as heads_kernel (msw_heads.cu):
//     hid = relu(fp16(A . W1^T + b1))   [rows x 2C],   out_h = fp16(hid_h . w2_h + b2_h),  h = policy, mine
// but the 128 x 2C accumulator of a row tile lives in TMEM instead of the register file, so the
// tensor pipe, the loads and the epilogue of three different tiles overlap inside one persistent CTA:
//   warp 0 (one lane)   TMA producer: W1 once, then the A tiles through a 3-stage ring
//                       (cp.async.bulk.tensor.2d, 128-byte swizzle, mbarrier complete_tx)
//   warp 1 (one lane)   MMA issuer: C/16 tcgen05.mma.kind::f16 (M = 128, N = 2C, K = 16) per tile into one of
//                       two TMEM accumulator stages; tcgen05.commit frees the smem stage / publishes the tile
//   warp 2              TMEM allocation (512 columns: 2 stages x 256) and release
//   warps 4-11          epilogue: tcgen05.ld of the thread's own row (TMEM lane = row), bias, fp16 rounding,
//                       ReLU and the C -> 1 dot product; warps 4-7 take the policy head, 8-11 the mine head
// K = C is not a multiple of the 64-element swizzle atom for C = 96: the second K block's box runs past the
// tensor's edge, TMA zero-fills it, and the issuer simply skips the k-steps that would multiply zeros.
#include "../../include/msw_b200.h"
#include "msw_error.h"
#include "msw_sm100.cuh"

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace msw {

constexpr int TC_ROWS = 128, TC_STAGES = 3, TC_THREADS = 384, TC_TMEM_COLS = 512, TC_ACC_STRIDE = 256;

template <int C>
struct TcCfg {
    static constexpr int KB = (C + 63) / 64;                 // 128-byte K blocks per operand tile
    static constexpr int N = 2 * C;                          // hidden units of both heads
    static constexpr int KSTEPS = C / 16;                    // tcgen05.mma instructions per tile
    static constexpr unsigned A_BLOCK = TC_ROWS * 128u, B_BLOCK = N * 128u;
    static constexpr unsigned A_STAGE = KB * A_BLOCK, B_BYTES = KB * B_BLOCK;
    static constexpr unsigned OFF_A = B_BYTES, OFF_B1 = OFF_A + TC_STAGES * A_STAGE, OFF_W2 = OFF_B1 + N * 4u;
    static constexpr unsigned OFF_BAR = OFF_W2 + N * 4u;     // full[3], empty[3], tmem_full[2], tmem_empty[2], b_full
    static constexpr unsigned OFF_TMEM = OFF_BAR + 11 * 8u;
    static constexpr unsigned BYTES = OFF_TMEM + 16u + 1024u;   // + slack to align the base to 1024 B
};

template <int C>
__global__ void __launch_bounds__(TC_THREADS, 1)
heads_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
                const __half *__restrict__ B1, const __half *__restrict__ W2, const __half *__restrict__ B2,
                __half *__restrict__ out_policy, __half *__restrict__ out_mine, long long R, long long tiles)
{
    using Cfg = TcCfg<C>;
    extern __shared__ unsigned char smem_dyn[];
    const unsigned base = (smem_u32(smem_dyn) + 1023u) & ~1023u;         // swizzled TMA tiles need 1024-byte alignment
    unsigned char *gen = smem_dyn + (base - smem_u32(smem_dyn));          // generic pointer to the same place
    const unsigned sB = base, sA = base + Cfg::OFF_A;
    float *s_b1 = reinterpret_cast<float *>(gen + Cfg::OFF_B1), *s_w2 = reinterpret_cast<float *>(gen + Cfg::OFF_W2);
    const unsigned bars = base + Cfg::OFF_BAR;
    auto full = [&](int s) { return bars + 8u * s; };
    auto empty = [&](int s) { return bars + 8u * (3 + s); };
    auto tfull = [&](int a) { return bars + 8u * (6 + a); };
    auto tempty = [&](int a) { return bars + 8u * (8 + a); };
    const unsigned bfull = bars + 8u * 10;
    volatile uint32_t *s_tmem = reinterpret_cast<volatile uint32_t *>(gen + Cfg::OFF_TMEM);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int s = 0; s < TC_STAGES; ++s) { mbar_init(full(s), 1); mbar_init(empty(s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull(a), 1); mbar_init(tempty(a), 8); }
        mbar_init(bfull, 1);
        mbar_fence_init();
    }
    if (warp == 2) tmem_alloc(base + Cfg::OFF_TMEM, TC_TMEM_COLS);
    if (warp >= 4)
        for (int q = tid - 128; q < Cfg::N; q += TC_THREADS - 128) {
            s_b1[q] = __half2float(B1[q]);
            s_w2[q] = __half2float(W2[q]);
        }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const unsigned tmem = *s_tmem;

    // warps 0 and 1 issue TMA / tcgen05 from one lane chosen by elect_one (msw_sm100.cuh says why not lane == 0)
    if (warp == 0) {
        if (elect_one()) {
        // ---- TMA producer
        mbar_expect_tx(bfull, Cfg::B_BYTES);
        for (int kb = 0; kb < Cfg::KB; ++kb) tma_load_2d(sB + kb * Cfg::B_BLOCK, &map_w, kb * 64, 0, bfull);
        unsigned it = 0;
        for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
            const unsigned s = it % TC_STAGES, ph = (it / TC_STAGES) & 1u;
            mbar_wait(empty(s), ph ^ 1u);
            mbar_expect_tx(full(s), Cfg::A_STAGE);
            for (int kb = 0; kb < Cfg::KB; ++kb)
                tma_load_2d(sA + s * Cfg::A_STAGE + kb * Cfg::A_BLOCK, &map_a, kb * 64, (int)(tile * TC_ROWS), full(s));
        }
        }
    } else if (warp == 1) {
        // ---- MMA issuer.  Instruction descriptor: D = F32 (bits 4-5 = 1), A = B = F16 (0), both K-major (0),
        // N >> 3 at bits 17-22, M >> 4 at bits 24-28.
        constexpr unsigned idesc = (1u << 4) | ((unsigned)(Cfg::N >> 3) << 17) | ((unsigned)(TC_ROWS >> 4) << 24);
        mbar_wait(bfull, 0);
        unsigned it = 0;
        for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
            const unsigned s = it % TC_STAGES, ph = (it / TC_STAGES) & 1u, as = it & 1u, aph = (it >> 1) & 1u;
            mbar_wait(tempty(as), aph ^ 1u);
            mbar_wait(full(s), ph);
            tcgen05_fence_after();
            const unsigned d = tmem + as * TC_ACC_STRIDE;
            if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < Cfg::KSTEPS; ++ks) {
                const int kb = ks / 4, k = ks % 4;                          // 4 k-steps of 32 bytes per swizzle atom
                const uint64_t da = umma_desc<128>(sA + s * Cfg::A_STAGE + kb * Cfg::A_BLOCK) + (uint64_t)(2 * k);
                const uint64_t db = umma_desc<128>(sB + kb * Cfg::B_BLOCK) + (uint64_t)(2 * k);
                umma_f16(d, da, db, idesc, ks > 0 ? 1u : 0u);
            }
            umma_commit(empty(s));           // the smem stage is free once these MMAs have read it
            umma_commit(tfull(as));          // ... and the accumulator is complete
            }
            __syncwarp();
        }
    } else if (warp >= 4) {
        // ---- epilogue: thread = one row of the tile (TMEM lane), one head per warpgroup
        const int q = warp & 3, head = (warp - 4) >> 2;
        const float b2 = __half2float(B2[head]);
        __half *__restrict__ out = head == 0 ? out_policy : out_mine;
        const float *b1 = s_b1 + head * C, *w2 = s_w2 + head * C;
        unsigned it = 0;
        for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
            const unsigned as = it & 1u, aph = (it >> 1) & 1u;
            mbar_wait(tfull(as), aph);
            tcgen05_fence_after();
            const unsigned taddr = tmem + as * TC_ACC_STRIDE + head * C + ((unsigned)(q * 32) << 16);
            float sum = 0.0f;
#pragma unroll
            for (int c0 = 0; c0 < C; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(taddr + c0, v);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 32; j += 2) {
                    // hid = relu(fp16(acc + b1)) for two columns at once, then fp32 dot with w2
                    const __half2 h = __hmax2(__floats2half2_rn(__uint_as_float(v[j]) + b1[c0 + j],
                                                                __uint_as_float(v[j + 1]) + b1[c0 + j + 1]),
                                              __float2half2_rn(0.0f));
                    const float2 f = __half22float2(h);
                    sum = fmaf(f.y, w2[c0 + j + 1], fmaf(f.x, w2[c0 + j], sum));
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty(as));
            const long long row = tile * TC_ROWS + q * 32 + lane;
            if (row < R) out[row] = __float2half_rn(sum + b2);
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 2) {
        tcgen05_fence_after();
        tmem_dealloc(tmem, TC_TMEM_COLS);
    }
}

// fp16 [rows][C] row-major, box = [box_rows][64 elements = 128 bytes], 128-byte swizzle, zero fill past the edges
static bool tc_make_map(CUtensorMap *m, const void *basep, int64_t rows, int C, int box_rows)
{
    const cuuint64_t dims[2] = {(cuuint64_t)C, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)C * 2};
    const cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
    return encode_tiled(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, basep, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B) == CUDA_SUCCESS;
}

template <int C>
static int launch_heads_tc(const void *a16, const void *w1, const void *b1, const void *w2, const void *b2,
                           void *out_policy, void *out_mine, int64_t R, cudaStream_t stream)
{
    using Cfg = TcCfg<C>;
    CUtensorMap ma, mw;
    if (!tc_make_map(&ma, a16, R, C, TC_ROWS) || !tc_make_map(&mw, w1, Cfg::N, C, Cfg::N))
        return fail(MSW_ERR_ARG, "msw_cell_heads: cuTensorMapEncodeTiled failed (rows=%lld C=%d)", (long long)R, C);
    MSW_SET_MAX_SMEM(heads_tc_kernel<C>, Cfg::BYTES);
    const int sms = sm_count();
    const long long tiles = (R + TC_ROWS - 1) / TC_ROWS;
    const long long grid = tiles < sms ? tiles : sms;                   // persistent, one CTA (all 512 TMEM columns) per SM
    heads_tc_kernel<C><<<(unsigned)grid, TC_THREADS, Cfg::BYTES, stream>>>(
        ma, mw, (const __half *)b1, (const __half *)w2, (const __half *)b2, (__half *)out_policy, (__half *)out_mine,
        (long long)R, tiles);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

// Entry used by msw_cell_heads (msw_heads.cu).  Returns -1 when this path does not apply (C, alignment, driver).
int heads_tc_launch(int C, const void *a16, const void *w1, const void *b1, const void *w2, const void *b2,
                    void *out_policy, void *out_mine, int64_t R, cudaStream_t stream)
{
    if (!tensor_map_encoder_available() || R > 0x7fffffffLL) return -1;
    switch (C) {
    case 64: return launch_heads_tc<64>(a16, w1, b1, w2, b2, out_policy, out_mine, R, stream);
    case 96: return launch_heads_tc<96>(a16, w1, b1, w2, b2, out_policy, out_mine, R, stream);
    case 128: return launch_heads_tc<128>(a16, w1, b1, w2, b2, out_policy, out_mine, R, stream);
    default: return -1;
    }
}

}  // namespace msw
