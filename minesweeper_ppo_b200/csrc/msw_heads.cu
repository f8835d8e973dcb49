// msw_heads.cu -- the two per-cell heads of the rollout forward in one kernel.
//
// CNNResidualPolicy ends in two 1x1-conv heads over the trunk activation f
// (minesweeper/models/cnn_residual.py:57-62, 73-77, 87-94):
//     policy logit = conv1x1_{C->1}( relu( conv1x1_{C->C}(f) ) )      per cell
//     mine logit   = conv1x1_{C->1}( relu( conv1x1_{C->C}(f) ) )      per cell (own weights)
// On the NHWC activation a 1x1 conv is a row-wise linear map, so both heads are
//     hid = relu(A . W1^T + b1)   [R x 2C],   out = hid . W2 (block diagonal) + b2   [R x 2]
// with R = n*H*W rows.  As library GEMMs the [R x 2C] hidden tensor (805 MB at 8,192 boards)
// is written, re-read by an eager ReLU and re-read by a 2-column GEMM (0.79 ms per forward,
// profiles/r01e_fused_forward_profile.txt).  Here it never leaves the registers: a CTA stages
// 128 rows of A (cp.async, double buffered) next to W1 in shared memory, warp (wm, wn) forms the
// 32 x C block of head wn with mma.sync m16n8k16 (fp16 in, fp32 accumulate), and the epilogue
// applies bias + fp16 rounding + ReLU (the rounding points of the autocast reference:
// train_rl.py:222) and the C->1 dot product in place.  HBM traffic: A once (2C bytes per row)
// plus 4 bytes of output per row.
#include "../../include/msw_b200.h"
#include "msw_error.h"
#include "msw_sm100.cuh"

#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

namespace msw {

constexpr int HEADS_ROWS = 128;     // rows of A per CTA tile
constexpr int HEADS_THREADS = 256;  // 8 warps: 4 along the rows x 2 heads

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void *smem)
{
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(smem)));
}
__device__ __forceinline__ void mma_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int C>
struct HeadsSmem {
    static constexpr int LD = C + 8;                 // padded row (halves): 16-byte aligned, odd multiple of 16 B
    __half w[2 * C][LD];                             // W1, row = hidden unit (policy units first, then mine units)
    __half a[2][HEADS_ROWS][LD];                     // two A tiles
    float b1[2 * C];
    float w2[2 * C];
};

// C <= 96: 96 accumulator registers, ~95 KB of shared memory -> two CTAs per SM; C = 128: one.
template <int C>
__global__ void __launch_bounds__(HEADS_THREADS, C <= 96 ? 2 : 1)
heads_kernel(const __half *__restrict__ A, const __half *__restrict__ W1, const __half *__restrict__ B1,
             const __half *__restrict__ W2, const __half *__restrict__ B2, __half *__restrict__ out_policy,
             __half *__restrict__ out_mine, long long R, long long tiles)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    HeadsSmem<C> &S = *reinterpret_cast<HeadsSmem<C> *>(smem_raw);
    constexpr int CH = C / 8;                        // 16-byte chunks per row
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp & 3, wn = warp >> 2;
    const int g = lane >> 2, t = lane & 3;

    auto stage_a = [&](long long tile, int buf) {
        const long long row0 = tile * HEADS_ROWS;
        for (int q = tid; q < HEADS_ROWS * CH; q += HEADS_THREADS) {
            const int r = q / CH, c = q % CH;
            long long row = row0 + r;
            if (row >= R) row = R - 1;               // tail rows repeat the last row; their results are not stored
            const __half *src = A + row * C + c * 8;
            cp_async16(smem_u32(&S.a[buf][r][c * 8]), src);
        }
    };

    long long tile = blockIdx.x;
    if (tile >= tiles) return;
    for (int q = tid; q < 2 * C * CH; q += HEADS_THREADS) {
        const __half *src = W1 + (long long)(q / CH) * C + (q % CH) * 8;
        cp_async16(smem_u32(&S.w[q / CH][(q % CH) * 8]), src);
    }
    stage_a(tile, 0);
    cp_async_commit();
    for (int q = tid; q < 2 * C; q += HEADS_THREADS) {
        S.b1[q] = __half2float(B1[q]);
        S.w2[q] = __half2float(W2[q]);
    }
    const float b2 = __half2float(B2[wn]);
    __half *__restrict__ out = wn == 0 ? out_policy : out_mine;

    int buf = 0;
    for (; tile < tiles; tile += gridDim.x, buf ^= 1) {
        const long long next = tile + gridDim.x;
        if (next < tiles) stage_a(next, buf ^ 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();                             // tile `buf` (and, the first time, W1 / b1 / w2) is visible

        float acc[2][C / 8][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int nt = 0; nt < C / 8; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[mt][nt][e] = 0.0f;

#pragma unroll
        for (int kk = 0; kk < C / 16; ++kk) {
            uint32_t af[2][4];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
                ldmatrix_x4(af[mt], &S.a[buf][wm * 32 + mt * 16 + (lane & 15)][kk * 16 + (lane >> 4) * 8]);
#pragma unroll
            for (int np = 0; np < C / 16; ++np) {
                // one x4 load = the B fragments of two adjacent 8-column tiles
                uint32_t bf[4];
                ldmatrix_x4(bf, &S.w[wn * C + np * 16 + (lane & 7) + ((lane >> 4) << 3)][kk * 16 + ((lane >> 3) & 1) * 8]);
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    mma_16816(acc[mt][2 * np], af[mt], bf[0], bf[1]);
                    mma_16816(acc[mt][2 * np + 1], af[mt], bf[2], bf[3]);
                }
            }
        }

        // epilogue: hid = relu(fp16(acc + b1)); out = fp16(sum_c hid_c * w2_c + b2)
        float part[2][2] = {{0.0f, 0.0f}, {0.0f, 0.0f}};       // [m-tile][row g / row g+8]
#pragma unroll
        for (int nt = 0; nt < C / 8; ++nt) {
            const int c = wn * C + nt * 8 + 2 * t;
            const float bb0 = S.b1[c], bb1 = S.b1[c + 1], ww0 = S.w2[c], ww1 = S.w2[c + 1];
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
                const float h0 = fmaxf(__half2float(__float2half_rn(acc[mt][nt][0] + bb0)), 0.0f);
                const float h1 = fmaxf(__half2float(__float2half_rn(acc[mt][nt][1] + bb1)), 0.0f);
                const float h2 = fmaxf(__half2float(__float2half_rn(acc[mt][nt][2] + bb0)), 0.0f);
                const float h3 = fmaxf(__half2float(__float2half_rn(acc[mt][nt][3] + bb1)), 0.0f);
                part[mt][0] = fmaf(h1, ww1, fmaf(h0, ww0, part[mt][0]));
                part[mt][1] = fmaf(h3, ww1, fmaf(h2, ww0, part[mt][1]));
            }
        }
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                float v = part[mt][hh];
                v += __shfl_xor_sync(0xffffffffu, v, 1);
                v += __shfl_xor_sync(0xffffffffu, v, 2);
                const long long row = tile * HEADS_ROWS + wm * 32 + mt * 16 + hh * 8 + g;
                if (t == 0 && row < R) out[row] = __float2half_rn(v + b2);
            }
        __syncthreads();                             // everyone is done with `buf` before it is refilled
    }
    cp_async_wait<0>();
}

template <int C>
static int launch_heads(const void *a16, const void *w1, const void *b1, const void *w2, const void *b2,
                        void *out_policy, void *out_mine, int64_t R, cudaStream_t stream)
{
    const size_t smem = sizeof(HeadsSmem<C>);
    MSW_SET_MAX_SMEM(heads_kernel<C>, smem);
    const int sms = sm_count();
    const long long tiles = (R + HEADS_ROWS - 1) / HEADS_ROWS;
    const long long resident = (C <= 96 ? 2LL : 1LL) * sms;             // persistent grid, one wave
    const long long grid = tiles < resident ? tiles : resident;
    heads_kernel<C><<<(unsigned)grid, HEADS_THREADS, smem, stream>>>(
        (const __half *)a16, (const __half *)w1, (const __half *)b1, (const __half *)w2, (const __half *)b2,
        (__half *)out_policy, (__half *)out_mine, (long long)R, tiles);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

// tcgen05 / TMEM implementation of the same operation (msw_heads_tc.cu); -1 = not applicable
int heads_tc_launch(int C, const void *a16, const void *w1, const void *b1, const void *w2, const void *b2,
                    void *out_policy, void *out_mine, int64_t R, cudaStream_t stream);

}  // namespace msw

extern "C" int msw_cell_heads(const void *a16, const void *w1, const void *b1, const void *w2, const void *b2,
                              void *out_policy, void *out_mine, int64_t rows, int32_t C, void *stream)
{
    using namespace msw;
    if (!a16 || !w1 || !b1 || !w2 || !b2 || !out_policy || !out_mine)
        return fail(MSW_ERR_NULL, "msw_cell_heads: NULL pointer");
    if (rows < 0) return fail(MSW_ERR_BAD_SHAPE, "msw_cell_heads: rows=%lld", (long long)rows);
    if ((((uintptr_t)a16 | (uintptr_t)w1) & 15u) != 0)
        return fail(MSW_ERR_ALIGN, "msw_cell_heads: a16 and w1 must be 16-byte aligned");
    if (rows == 0) return MSW_OK;
    cudaStream_t s = (cudaStream_t)stream;
    // one kernel per width: tcgen05 (msw_heads_tc.cu) for C = 64 / 96 / 128, whose N = 2C fills an MMA tile;
    // the mma.sync kernel of this file only for C = 32
    if (C == 32) return launch_heads<32>(a16, w1, b1, w2, b2, out_policy, out_mine, rows, s);
    const int rc = heads_tc_launch(C, a16, w1, b1, w2, b2, out_policy, out_mine, rows, s);
    if (rc >= 0) return rc;
    return fail(MSW_ERR_BAD_SHAPE, "msw_cell_heads: C=%d (supported: 32, 64, 96, 128)", C);
}
