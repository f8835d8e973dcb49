// msw_sampler.cu -- fused masked categorical sampler (SURVEY.md section 8, row f1).
//
// Replaces the per-step ATen sequence of the reference collector (train_rl.py:229-235):
//     logits = logits.masked_fill(~mask, neg_inf)         neg_inf = -1e4 (fp16/bf16) / -1e9 (fp32)
//     dist = Categorical(logits=logits); actions = dist.sample(); logp = dist.log_prob(actions)
// plus the int64 -> int32 action conversion of train_rl.py:239, in ONE launch that reads the mask
// the env kernel just wrote and writes actions (int64 for the buffer, int32 for the env) and
// log-probabilities straight into the rollout buffer.
//
// One warp per row.  Arithmetic is fp32 on the (possibly half) logits: log-softmax is exact to
// fp32 rounding, sampling is inverse-CDF over the row in index order with one Philox uniform per
// (seed, global row, step).  torch's own RNG stream is not reproduced (it is not part of any
// parity contract); the distribution and the log-probabilities are.
#include "../../include/msw_b200.h"
#include "msw_common.cuh"
#include "msw_error.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace msw {


template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ float round_to(float v);     // fill value as T stores it
template <> __device__ __forceinline__ float round_to<float>(float v) { return v; }
template <> __device__ __forceinline__ float round_to<__half>(float v) { return __half2float(__float2half_rn(v)); }
template <> __device__ __forceinline__ float round_to<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

template <typename T, int MAXC>
__global__ void __launch_bounds__(128)
masked_sample_kernel(const T *__restrict__ logits, uint8_t *__restrict__ mask, long long n, int A,
                     float neg_inf_in, uint32_t k0, uint32_t k1, uint32_t step_lo, uint32_t step_hi,
                     const uint32_t *__restrict__ epoch, long long row_id_base, long long *__restrict__ a64, int32_t *__restrict__ a32,
                     float *__restrict__ logp)
{
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    const int chunk = (A + 31) >> 5;                       // contiguous cells per lane (<= MAXC)
    const float neg_inf = round_to<T>(neg_inf_in);
    const int lo = lane * chunk;
    const T *lrow = logits + row * (long long)A;
    uint8_t *mrow = mask + row * (long long)A;

    uint32_t mb = 0u;                                       // this lane's mask bits
#pragma unroll
    for (int j = 0; j < MAXC; ++j)
        if (j < chunk && lo + j < A && mrow[lo + j]) mb |= 1u << j;
    // A row without a single legal action becomes all-legal, in the stored mask too (the collector's guard,
    // train_rl.py:166-168 / 263-265; unreachable through the env, which resets finished boards).
    const bool none = __ballot_sync(FULL, mb != 0u) == 0u;
    if (none) {
        mb = 0xffffffffu;
#pragma unroll
        for (int j = 0; j < MAXC; ++j)
            if (j < chunk && lo + j < A) mrow[lo + j] = 1;
    }
    float v[MAXC];
    float mx = -3.0e38f;
#pragma unroll
    for (int j = 0; j < MAXC; ++j) {
        if (j < chunk) {
            const int i = lo + j;
            float x = -3.0e38f;
            if (i < A) x = (mb >> j & 1u) ? to_f32<T>(lrow[i]) : neg_inf;     // masked_fill (train_rl.py:232)
            v[j] = x;
            mx = fmaxf(mx, x);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, o));

    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < MAXC; ++j) {
        if (j < chunk) {
            const float e = (lo + j < A) ? expf(v[j] - mx) : 0.0f;
            v[j] = e;
            s += e;
        }
    }
    float incl = s;                                        // inclusive scan of the lane sums
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
    }
    const float total = __shfl_sync(FULL, incl, 31);

    const unsigned long long rid = (unsigned long long)(row_id_base + row);
    uint32_t w[4];
    // `epoch` (device counter, nullable) lets a captured CUDA graph draw fresh numbers on every replay
    const uint32_t hi = step_hi + (epoch ? *epoch : 0u);
    philox4x32_10(k0, k1 ^ 0x53414d50u, (uint32_t)rid, (uint32_t)(rid >> 32), step_lo, hi, w);
    // (0, 1], 24 bits: once w0 >> 8 >= 2^23 the half is lost to rounding, so w0 >> 8 == 0xFFFFFF gives exactly 1
    const float u = ((float)(w[0] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float target = u * total;

    // first lane with mass whose running total exceeds the target.  The float32 scan is not monotone across lanes:
    // an empty lane's `incl` can round one ulp above the lanes before it (or above `total`), and a target in that
    // gap must not land there -- its first cell is masked, or past the row when 32 does not divide A.
    // Rounding can leave no such lane (u == 1 among them) -> last non-empty lane.
    const unsigned over = __ballot_sync(FULL, incl > target && s > 0.0f);
    const unsigned nonempty = __ballot_sync(FULL, s > 0.0f);
    const int owner = over ? (__ffs(over) - 1) : (31 - __clz(nonempty | 1u));
    int action = 0;
    float la = 0.0f;
    if (lane == owner) {
        float run = incl - s;
        int pick = -1, last_pos = -1;
#pragma unroll
        for (int j = 0; j < MAXC; ++j) {
            if (j < chunk && lo + j < A) {
                run += v[j];
                if (v[j] > 0.0f) last_pos = j;
                if (pick < 0 && v[j] > 0.0f && run > target) pick = j;
            }
        }
        if (pick < 0) pick = last_pos < 0 ? 0 : last_pos;
        action = lo + pick;
    }
    action = __shfl_sync(FULL, action, owner);
    if (lane == 0) {
        // log_prob = logit - max - log(sum exp(logit - max))  (Categorical normalisation)
        const float x = (none || mrow[action]) ? to_f32<T>(lrow[action]) : neg_inf;
        la = (x - mx) - logf(total);
        if (a64) a64[row] = action;
        if (a32) a32[row] = action;
        if (logp) logp[row] = la;
    }
}

}  // namespace msw

extern "C" int msw_masked_sample(const void *logits, int32_t logits_dtype, uint8_t *mask, int64_t n,
                                 int32_t A, uint64_t seed, uint64_t step_index, const uint32_t *epoch,
                                 int64_t row_id_base,
                                 int64_t *actions64, int32_t *actions32, float *logp, void *stream)
{
    using namespace msw;
    if (!logits || !mask) return fail(MSW_ERR_NULL, "msw_masked_sample: logits/mask is NULL");
    if (!actions64 && !actions32) return fail(MSW_ERR_NULL, "msw_masked_sample: no action output");
    if (A < 1 || A > MSW_MAX_CELLS || n < 0) return fail(MSW_ERR_BAD_SHAPE, "msw_masked_sample: A=%d n=%lld", A, (long long)n);
    if (n == 0) return MSW_OK;
    const unsigned grid = (unsigned)((n + 3) / 4);
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    const uint32_t s0 = (uint32_t)step_index, s1 = (uint32_t)(step_index >> 32);
    cudaStream_t st = (cudaStream_t)stream;
    long long *a64 = reinterpret_cast<long long *>(actions64);
    const int chunk = (A + 31) / 32;
#define MSW_LAUNCH_SAMPLER(T, NEG)                                                                              \
    do {                                                                                                        \
        if (chunk <= 8)                                                                                         \
            masked_sample_kernel<T, 8><<<grid, 128, 0, st>>>((const T *)logits, mask, n, A, NEG, k0, k1, s0, s1, \
                                                             epoch, row_id_base, a64, actions32, logp);               \
        else if (chunk <= 16)                                                                                   \
            masked_sample_kernel<T, 16><<<grid, 128, 0, st>>>((const T *)logits, mask, n, A, NEG, k0, k1, s0,   \
                                                              s1, epoch, row_id_base, a64, actions32, logp);          \
        else                                                                                                    \
            masked_sample_kernel<T, 32><<<grid, 128, 0, st>>>((const T *)logits, mask, n, A, NEG, k0, k1, s0,   \
                                                              s1, epoch, row_id_base, a64, actions32, logp);          \
    } while (0)
    switch (logits_dtype) {                       // fill constants of train_rl.py:229-232
    case 0: MSW_LAUNCH_SAMPLER(float, -1e9f); break;
    case 1: MSW_LAUNCH_SAMPLER(__half, -1e4f); break;
    case 2: MSW_LAUNCH_SAMPLER(__nv_bfloat16, -1e4f); break;
    default:
        return fail(MSW_ERR_ARG, "msw_masked_sample: logits_dtype %d (0 f32, 1 f16, 2 bf16)", logits_dtype);
    }
#undef MSW_LAUNCH_SAMPLER
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}
