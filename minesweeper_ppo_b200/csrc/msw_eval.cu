// msw_eval.cu -- device-resident greedy evaluator (DESIGN.md section 4.9).
//
// Replaces the per-step host work of eval.evaluate_vec (eval.py:265-511) that the NumPy-API mirror
// (evaluate.py::evaluate_vec) still does on the CPU:
//   masked_argmax_kernel   logits.masked_fill(~mask, -1e9).argmax(-1) with the empty-row guard
//                          (eval.py:330-340), int32 actions for the env;
//   eval_pre_kernel        the per-env loop BEFORE the step (eval.py:350-398): invalid picks, the `safe`
//                          test, subset-rule hit / guess, avoidability bookkeeping and the belief-pair
//                          selection plane, from the msw_forced_subset / msw_avoidability arrays;
//   eval_post_kernel       the per-env loop AFTER the step (eval.py:405-428): progress, wins, steps, the
//                          first-finished-episode accounting and the max_steps cutoff.
// Counters are int64 and updated with integer atomics (shared memory per block, then one global atomic per
// block and counter), so the totals do not depend on the order in which envs are processed.
#include "../../include/msw_b200.h"
#include "msw_common.cuh"
#include "msw_error.h"

#include <cuda_runtime.h>
#include <stdint.h>

namespace msw {

// torch's argmax order (ATen GreaterOrNan): NaN beats everything, the first NaN wins; otherwise the larger
// value, and the smaller index on ties.
__device__ __forceinline__ bool argmax_better(float v, int i, float bv, int bi)
{
    const bool vn = v != v, bn = bv != bv;
    if (vn) return !bn || i < bi;
    if (bn) return false;
    return v > bv || (v == bv && i < bi);
}

__global__ void __launch_bounds__(128)
masked_argmax_kernel(const float *__restrict__ logits, uint8_t *__restrict__ mask, long long n, int A,
                     int32_t *__restrict__ actions)
{
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    const float *lrow = logits + row * (long long)A;
    uint8_t *mrow = mask + row * (long long)A;

    bool any = false;
    for (int i = lane; i < A; i += 32) any |= mrow[i] != 0;
    // A row without a single legal action becomes all-legal, in the stored mask too (eval.py:336-338).
    const bool none = __ballot_sync(FULL, any) == 0u;
    if (none)
        for (int i = lane; i < A; i += 32) mrow[i] = 1;

    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = lane; i < A; i += 32) {
        const float x = (none || mrow[i]) ? lrow[i] : -1e9f;     // masked cells still compete at -1e9
        if (argmax_better(x, i, bv, bi)) { bv = x; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(FULL, bv, o);
        const int oi = __shfl_xor_sync(FULL, bi, o);
        if (argmax_better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) actions[row] = bi;
}

// Block-level accumulation: lanes 0 of the warps add into shared int64 slots, then one global atomic per
// non-zero slot.  Integer adds commute, so the result is independent of the schedule.
template <int K>
struct BlockCounters {
    unsigned long long *s;
    __device__ void init()
    {
        for (int k = threadIdx.x; k < K; k += blockDim.x) s[k] = 0ull;
        __syncthreads();
    }
    __device__ void add(int k, long long v)
    {
        if (v) atomicAdd(&s[k], (unsigned long long)v);
    }
    __device__ void flush(long long *g)
    {
        __syncthreads();
        for (int k = threadIdx.x; k < K; k += blockDim.x)
            if (s[k]) atomicAdd(reinterpret_cast<unsigned long long *>(g + k), s[k]);
    }
};

__device__ __forceinline__ bool bit_of(const uint32_t *row, int cell)
{
    return (row[cell >> 5] >> (cell & 31)) & 1u;
}

__global__ void __launch_bounds__(256)
eval_pre_kernel(int H, int W, int wpb, long long n, long long batch_size, const uint32_t *__restrict__ mines,
                const uint32_t *__restrict__ revealed, const uint32_t *__restrict__ flags,
                const int32_t *__restrict__ meta, const int32_t *__restrict__ actions,
                const uint8_t *__restrict__ mask, const uint32_t *__restrict__ subset_bits,
                const uint32_t *__restrict__ safe_bits, const int16_t *__restrict__ comp_of_cell,
                const int16_t *__restrict__ comp_size, const uint8_t *__restrict__ avoid_flags,
                const uint8_t *__restrict__ counted, uint8_t *__restrict__ ep_unavoidable,
                uint8_t *__restrict__ belief_sel, long long *__restrict__ counters, long long step_index)
{
    __shared__ unsigned long long s_acc[MSW_EVAL_PRE_COUNTERS];
    BlockCounters<MSW_EVAL_PRE_COUNTERS> acc{s_acc};
    acc.init();
    const int lane = threadIdx.x & 31;
    const long long i = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int HW = H * W;
    if (i < n) {
        const int cell = actions[i];
        if (lane == 0 && !mask[i * HW + cell]) acc.add(MSW_EVAL_INVALID, 1);      // over ALL envs (eval.py:339-340)
        const bool live = !counted[i] && i < batch_size;
        const uint32_t *mrow = mines + i * wpb, *rrow = revealed + i * wpb;
        const uint32_t *frow = flags ? flags + i * wpb : nullptr;
        if (belief_sel) {              // 0: not a belief pair; 1 + mine: unknown cell of a live env (eval.py:352-358)
            uint8_t *srow = belief_sel + i * HW;
            for (int c = lane; c < HW; c += 32) {
                uint8_t v = 0;
                if (live && !bit_of(rrow, c) && !(frow && bit_of(frow, c))) v = (uint8_t)(1 + bit_of(mrow, c));
                srow[c] = v;
            }
        }
        if (live) {
            const bool safe = !bit_of(mrow, cell);
            if (lane == 0) {                                                       // eval.py:362-379
                if (bit_of(subset_bits + i * wpb, cell)) {
                    acc.add(MSW_EVAL_FORCED_STEPS, 1); acc.add(MSW_EVAL_FORCED_CORRECT, safe);
                } else {
                    acc.add(MSW_EVAL_GUESS_ATTEMPTS, 1); acc.add(MSW_EVAL_GUESS_SUCCESS, safe);
                }
            }
            if (meta[i * 4 + 0]) {                                                 // first_click_done: eval.py:381-398
                const int fl = avoid_flags[i];
                const int16_t *cs = comp_size + i * HW;
                long long csum = 0, ccnt = 0;
                for (int c = lane; c < HW; c += 32) {
                    const int v = cs[c];
                    if (v > 0) { csum += v; ++ccnt; }
                }
                int nsafe = 0;
                for (int w = lane; w < wpb; w += 32) nsafe += __popc(safe_bits[i * wpb + w]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    csum += __shfl_xor_sync(FULL, csum, o);
                    ccnt += __shfl_xor_sync(FULL, ccnt, o);
                    nsafe += __shfl_xor_sync(FULL, nsafe, o);
                }
                if (lane == 0) {
                    if (fl & 8)             // the exact search ran out of budget: the reference would raise here
                        atomicMin(reinterpret_cast<unsigned long long *>(counters + MSW_EVAL_ERROR_KEY),
                                  (unsigned long long)(step_index * n + i));
                    acc.add(MSW_EVAL_COMP_SIZE_SUM, csum); acc.add(MSW_EVAL_COMP_COUNT, ccnt);
                    // chosen-cell fields of AvoidabilityResult (avoidability.py:41-49)
                    bool chosen_safe = false;
                    int chosen_size = -1;
                    if (fl & 4) {
                        if (fl & 2) {
                            const int lab = comp_of_cell[i * HW + cell];
                            if (lab >= 0) {
                                chosen_size = comp_size[i * HW + lab];
                                chosen_safe = bit_of(safe_bits + i * wpb, cell);
                            }
                        } else if (!bit_of(rrow, cell)) {
                            chosen_size = 1;
                        }
                    }
                    if (chosen_size >= 0) { acc.add(MSW_EVAL_CHOSEN_SIZE_SUM, chosen_size); acc.add(MSW_EVAL_CHOSEN_COUNT, 1); }
                    acc.add(MSW_EVAL_REVEAL_TOTAL, 1);
                    if (fl & 1) {
                        acc.add(MSW_EVAL_SAFE_OPTION_TOTAL, 1);
                        acc.add(MSW_EVAL_SAFE_CELLS, nsafe);
                        acc.add(chosen_safe ? MSW_EVAL_SAFE_OPTION_HITS : MSW_EVAL_SAFE_OPTION_MISSES, 1);
                    } else {
                        acc.add(MSW_EVAL_FORCED_GUESS_TOTAL, 1);
                        acc.add(MSW_EVAL_FORCED_GUESS_SUCCESS, safe);
                        ep_unavoidable[i] = 1;
                    }
                }
            }
        }
    }
    acc.flush(counters);
}

__global__ void __launch_bounds__(256)
eval_post_kernel(long long n, const uint8_t *__restrict__ done, const int8_t *__restrict__ outcome,
                 const int32_t *__restrict__ new_reveals, uint8_t *__restrict__ counted,
                 int32_t *__restrict__ step_counter, const uint8_t *__restrict__ ep_unavoidable, int max_steps,
                 long long *__restrict__ counters, int32_t *__restrict__ finished)
{
    __shared__ unsigned long long s_acc[MSW_EVAL_COUNTERS];
    BlockCounters<MSW_EVAL_COUNTERS> acc{s_acc};
    acc.init();
    __shared__ int s_fin;
    if (threadIdx.x == 0) s_fin = 0;
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {                                                  // eval.py:405-428, over ALL envs
        int steps = step_counter[i] + 1;
        bool c = counted[i];
        int fin = 0;
        if (!c) acc.add(MSW_EVAL_NEW_REVEALS, new_reveals[i]);
        if (!c && done[i]) {
            acc.add(MSW_EVAL_WINS, outcome[i] == 1);
            acc.add(MSW_EVAL_TOTAL_STEPS, steps);
            acc.add(MSW_EVAL_FORCED_GUESS_EPISODES, ep_unavoidable[i] != 0);
            steps = 0; c = true; fin = 1;
        }
        if (!c && 0 < max_steps && max_steps <= steps) {
            acc.add(MSW_EVAL_TOTAL_STEPS, steps);
            steps = 0; c = true; fin = 1;
        }
        step_counter[i] = steps;
        if (fin) { counted[i] = 1; atomicAdd(&s_fin, 1); }
    }
    acc.flush(counters);
    if (threadIdx.x == 0 && s_fin) atomicAdd(finished, s_fin);
}

}  // namespace msw

extern "C" int msw_masked_argmax(const float *logits, uint8_t *mask, int64_t n, int32_t A, int32_t *actions,
                                 void *stream)
{
    using namespace msw;
    if (!logits || !mask || !actions) return fail(MSW_ERR_NULL, "msw_masked_argmax: logits/mask/actions is NULL");
    if (A < 1 || A > MSW_MAX_CELLS || n < 0) return fail(MSW_ERR_BAD_SHAPE, "msw_masked_argmax: A=%d n=%lld", A, (long long)n);
    if (n == 0) return MSW_OK;
    masked_argmax_kernel<<<(unsigned)((n + 3) / 4), 128, 0, (cudaStream_t)stream>>>(logits, mask, n, A, actions);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

extern "C" int msw_eval_pre_step(const msw_env_desc *desc, const msw_state *st, int64_t n, int64_t batch_size,
                                 const int32_t *actions, const uint8_t *mask, const uint32_t *subset_bits,
                                 const uint32_t *safe_bits, const int16_t *comp_of_cell, const int16_t *comp_size,
                                 const uint8_t *avoid_flags, const uint8_t *counted, uint8_t *ep_unavoidable,
                                 uint8_t *belief_sel, int64_t *counters, int64_t step_index, void *stream)
{
    using namespace msw;
    if (!desc || !st || !st->mines || !st->revealed || !st->meta || !actions || !mask || !subset_bits || !safe_bits ||
        !comp_of_cell || !comp_size || !avoid_flags || !counted || !ep_unavoidable || !counters)
        return fail(MSW_ERR_NULL, "msw_eval_pre_step: a required pointer is NULL");
    const int wpb = msw_words_per_board(desc->H, desc->W);
    if (wpb == 0 || n < 0 || batch_size < 0 || step_index < 0)
        return fail(MSW_ERR_BAD_SHAPE, "msw_eval_pre_step: H=%d W=%d n=%lld", desc->H, desc->W, (long long)n);
    if (n == 0) return MSW_OK;
    eval_pre_kernel<<<(unsigned)((n + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
        desc->H, desc->W, wpb, n, batch_size, st->mines, st->revealed, st->flags, st->meta, actions, mask, subset_bits,
        safe_bits, comp_of_cell, comp_size, avoid_flags, counted, ep_unavoidable, belief_sel,
        reinterpret_cast<long long *>(counters), step_index);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

extern "C" int msw_eval_post_step(int64_t n, const uint8_t *done, const int8_t *outcome, const int32_t *new_reveals,
                                  uint8_t *counted, int32_t *step_counter, const uint8_t *ep_unavoidable,
                                  int32_t max_steps, int64_t *counters, int32_t *finished, void *stream)
{
    using namespace msw;
    if (!done || !outcome || !new_reveals || !counted || !step_counter || !ep_unavoidable || !counters || !finished)
        return fail(MSW_ERR_NULL, "msw_eval_post_step: a required pointer is NULL");
    if (n < 0) return fail(MSW_ERR_BAD_SHAPE, "msw_eval_post_step: n=%lld", (long long)n);
    if (n == 0) return MSW_OK;
    eval_post_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        n, done, outcome, new_reveals, counted, step_counter, ep_unavoidable, max_steps,
        reinterpret_cast<long long *>(counters), finished);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}
