// msw_gae.cu -- RolloutBuffer.compute_gae (minesweeper/buffers.py:78-94) as one
// sm_100a kernel.
//
// The recurrence is serial in t and independent per env column, and the
// reference evaluates it in unfused IEEE fp32 in a fixed operation order, which
// this kernel reproduces bit for bit (__fmul_rn/__fadd_rn/__fsub_rn never
// contract into FMA):
//     nnt   = 1.0 - float(done[t])                                   (:89)
//     delta = (rewards[t] + (gamma * next_value) * nnt) - values[t]   (:90)
//     last  = delta + ((gamma*lam) * nnt) * last                      (:91)
//     returns = advantages + values                                   (:94)
// Storage is time-major [T][N] (buffers.py:81-83), so a row of 32 consecutive
// columns is one 128-byte line and a CTA owns 32 columns.  Only `last` carries a
// dependency from t+1 to t -- next_value is values[t+1], plain data -- so delta[t]
// is formed for all elements in parallel and the one warp that walks the chains
// does just FSEL / FMUL / FADD per step out of shared memory / registers.
// Two kernels share that arithmetic: gae_pipe_kernel (TMA slices through a
// shared-memory ring, warp-specialised; the default) and gae_kernel (plain
// coalesced loads, for ragged N the tensor maps cannot describe).  HBM-bound when
// there are many columns (17 B per transition), latency-bound at the reference's
// sizes, where the serial walk is the critical path.
#include "../../include/msw_b200.h"
#include "msw_error.h"
#include "msw_sm100.cuh"

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace msw {

constexpr int GAE_TC = 128;     // time rows per shared-memory chunk
constexpr int GAE_THREADS = 256;
// 32 env columns per CTA (one full 128-byte line per row).  16 columns -- twice the CTAs, so every SM
// has work at N = 8,192 -- was measured slower (18.4 vs 14.3 us, half-line requests) and removed.
constexpr int COLS = 32;

// Thread t loads column t % COLS of rows t / COLS, t / COLS + 256 / COLS, ...; the first COLS lanes of warp 0
// walk the chains.
__global__ void __launch_bounds__(GAE_THREADS)
gae_kernel(const float *__restrict__ rewards, const float *__restrict__ values,
           const uint8_t *__restrict__ dones, const float *__restrict__ last_values,
           float *__restrict__ adv, float *__restrict__ ret, long long T, long long N,
           float gamma, float gamma_lam, int prescaled)
{
    __shared__ float s_r[GAE_TC][COLS];     // rewards in, then delta, then advantages
    __shared__ float s_v[GAE_TC][COLS];
    __shared__ uint8_t s_d[GAE_TC][COLS];
    __shared__ float s_gvn[COLS];           // gamma * value of the row after this chunk's last one
    constexpr int RPP = GAE_THREADS / COLS;       // rows per pass of the whole CTA
    constexpr int RPT = GAE_TC / RPP;             // rows per thread and chunk

    const int c = threadIdx.x % COLS;
    const int rr = threadIdx.x / COLS;
    const long long col = (long long)blockIdx.x * COLS + c;
    const bool in = col < N;
    const bool chain = threadIdx.x < COLS;        // warp 0, first COLS lanes

    float last = 0.0f;                                          // buffers.py:86
    if (chain) {                                                // buffers.py:88 (t == T-1)
        const float lv = in ? last_values[col] : 0.0f;
        // prescaled: last_values already is gamma*last_value (fp16 bootstrap)
        s_gvn[c] = prescaled ? lv : __fmul_rn(gamma, lv);
    }

    for (long long t_hi = T; t_hi > 0; t_hi -= GAE_TC) {
        const long long t_lo = t_hi > GAE_TC ? t_hi - GAE_TC : 0;
        const int rows = (int)(t_hi - t_lo);
        // ---- load: every thread issues all of its (up to 3*RPT) loads before the first use, so a
        // CTA has its whole tile in flight at once (the kernel is latency-, not bandwidth-bound)
        {
            float r[RPT], v[RPT];
            uint8_t d[RPT];
#pragma unroll
            for (int k = 0; k < RPT; ++k) {
                const int i = rr + k * RPP;
                const bool ok = in && i < rows;
                const long long idx = (t_lo + i) * N + col;
                r[k] = ok ? __ldcs(rewards + idx) : 0.0f;
                v[k] = ok ? __ldcs(values + idx) : 0.0f;
                d[k] = ok ? __ldcs(dones + idx) : (uint8_t)0;
            }
#pragma unroll
            for (int k = 0; k < RPT; ++k) {
                const int i = rr + k * RPP;
                s_r[i][c] = r[k];
                s_v[i][c] = v[k];
                s_d[i][c] = d[k];
            }
        }
        __syncthreads();
        // ---- delta[t] = (r[t] + (gamma * v[t+1]) * nnt[t]) - v[t] for the thread's own elements
        // (buffers.py:88-90); each thread rewrites only the s_r entries it stored itself
#pragma unroll
        for (int k = 0; k < RPT; ++k) {
            const int i = rr + k * RPP;
            if (i < rows) {
                const float gv = i + 1 < rows ? __fmul_rn(gamma, s_v[i + 1][c]) : s_gvn[c];
                const float nn = s_d[i][c] ? 0.0f : 1.0f;
                s_r[i][c] = __fsub_rn(__fadd_rn(s_r[i][c], __fmul_rn(gv, nn)), s_v[i][c]);
            }
        }
        __syncthreads();
        // ---- chain: last = delta + ((gamma*lam) * nnt) * last (buffers.py:91), 8 rows per batch read
        // into registers ahead of the dependent arithmetic
        if (chain) {
            s_gvn[c] = __fmul_rn(gamma, s_v[0][c]);     // for the chunk before this one in time
            for (int hi = rows; hi > 0; hi -= 8) {
                float dl[8], gl[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int i = hi - 1 - k >= 0 ? hi - 1 - k : 0;
                    dl[k] = s_r[i][c];
                    gl[k] = s_d[i][c] ? 0.0f : gamma_lam;      // == gamma_lam * nnt exactly
                }
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int i = hi - 1 - k;
                    if (i >= 0) {
                        last = __fadd_rn(dl[k], __fmul_rn(gl[k], last));
                        s_r[i][c] = last;
                    }
                }
            }
        }
        __syncthreads();
        if (in) {
#pragma unroll
            for (int k = 0; k < RPT; ++k) {
                const int i = rr + k * RPP;
                if (i < rows) {
                    const long long idx = (t_lo + i) * N + col;
                    const float a = s_r[i][c];
                    __stcs(adv + idx, a);
                    __stcs(ret + idx, __fadd_rn(a, s_v[i][c]));
                }
            }
        }
        __syncthreads();        // the next chunk overwrites the tiles and reads s_gvn
    }
}

// ---------------------------------------------------------------------------
// TMA kernel (the default when N % 16 == 0 and the arrays are 16-byte aligned): the same arithmetic in [32 x 32]
// time slices through a 4-stage shared-memory ring, with the three kinds of work on different warps so that only
// the serial walk is on a CTA's critical path:
//   warp 4   (producer) keeps up to four slices in flight (one cp.async.bulk.tensor.2d per array and slice ->
//            `full` mbarriers; out-of-range rows / columns are zero-filled on load and clipped on store by the
//            tensor map, so ragged T and N need no predicates), streams finished slices out with TMA stores and
//            refills a stage as soon as its stores have read it;
//   warps 1-3 (delta)   form delta[t] for a slice as soon as it lands -- gamma*v[t+1] across a slice boundary comes
//            from a register they saved while the previous slice's values were still untouched -> `dd` mbarriers;
//   warp 0   (walk)     runs last = delta + c*last down the slice and forms returns = advantages + values in the
//            same pass (off the dependent chain) -> `done` mbarriers.
// Slices are processed newest-time-first; every operation and its order are those of gae_kernel above.
// Measured on one B200 (profiles/r02x_gae_ab.txt) against round 2's first TMA kernel, which moved whole [128 x 32]
// tiles load -> delta -> walk -> store with nothing overlapping inside a CTA (commit 9cc9c01): T=128, N=8,192
// 5.2 vs 7.0 us back to back, 12.3 vs 14.3 us cold; N=524,288 (HBM-bound) 186 vs 222 us = 6.13 vs 5.15 TB/s
// (0.94 vs 0.79 of the measured copy peak).  The mbarrier / TMA wrappers are in msw_sm100.cuh.
// ---------------------------------------------------------------------------
constexpr int PG_ROWS = 32, PG_COLS = 32, PG_STAGES = 4, PG_DWARPS = 3, PG_THREADS = (1 + PG_DWARPS + 1) * 32;

struct PipeStage {
    alignas(128) float r[PG_ROWS][PG_COLS];      // rewards in, delta, advantages out
    alignas(128) float v[PG_ROWS][PG_COLS];      // values in, returns out
    alignas(128) uint8_t d[PG_ROWS][PG_COLS];
};
struct PipeSmem {
    PipeStage st[PG_STAGES];
    alignas(8) unsigned long long full[PG_STAGES], dd[PG_STAGES], done[PG_STAGES];
};

template <int BATCH>
__global__ void __launch_bounds__(PG_THREADS, BATCH == PG_ROWS ? 1 : 5)
gae_pipe_kernel(const __grid_constant__ CUtensorMap m_rewards, const __grid_constant__ CUtensorMap m_values,
                const __grid_constant__ CUtensorMap m_dones, const __grid_constant__ CUtensorMap m_adv,
                const __grid_constant__ CUtensorMap m_ret, const float *__restrict__ last_values, long long T,
                long long N, float gamma, float gamma_lam, int prescaled)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    PipeSmem &S = *reinterpret_cast<PipeSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int col0 = blockIdx.x * PG_COLS;
    constexpr unsigned SLICE_BYTES = PG_ROWS * PG_COLS * (4 + 4 + 1);
    const int slices = (int)((T + PG_ROWS - 1) / PG_ROWS);      // slice j (processing order) = rows [(slices-1-j)*32, +32)

    if (tid == 0) {
        for (int s = 0; s < PG_STAGES; ++s) {
            mbar_init(smem_u32(&S.full[s]), 1);
            mbar_init(smem_u32(&S.dd[s]), PG_DWARPS * 32);
            mbar_init(smem_u32(&S.done[s]), 32);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == 1 + PG_DWARPS) {
        // ---- producer
        if (elect_one()) {
            // the store descriptors are first needed a few us into the kernel: fetch them now, off the critical path
            tma_prefetch(&m_adv);
            tma_prefetch(&m_ret);
            auto load = [&](int j) {
                PipeStage &st = S.st[j % PG_STAGES];
                const unsigned bar = smem_u32(&S.full[j % PG_STAGES]);
                const int row0 = (slices - 1 - j) * PG_ROWS;
                mbar_expect_tx(bar, SLICE_BYTES);
                tma_load_2d(smem_u32(&st.r[0][0]), &m_rewards, col0, row0, bar);
                tma_load_2d(smem_u32(&st.v[0][0]), &m_values, col0, row0, bar);
                tma_load_2d(smem_u32(&st.d[0][0]), &m_dones, col0, row0, bar);
            };
            for (int j = 0; j < slices && j < PG_STAGES; ++j) load(j);
            for (int j = 0; j < slices; ++j) {
                const int s = j % PG_STAGES;
                const unsigned ph = (unsigned)(j / PG_STAGES) & 1u;
                mbar_wait(smem_u32(&S.done[s]), ph);
                const int row0 = (slices - 1 - j) * PG_ROWS;
                tma_store_2d(&m_adv, col0, row0, smem_u32(&S.st[s].r[0][0]));
                tma_store_2d(&m_ret, col0, row0, smem_u32(&S.st[s].v[0][0]));
                bulk_commit();
                if (j + PG_STAGES < slices) {
                    bulk_wait_read<0>();                  // the stage's stores have read it
                    load(j + PG_STAGES);
                }
            }
            bulk_wait<0>();
        }
        return;
    }

    if (warp >= 1) {
        // ---- delta warps: warp w owns rows w-1, w+2, ... of every slice, lane = column
        const float lv = col0 + lane < N ? last_values[col0 + lane] : 0.0f;
        float gvn = prescaled ? lv : __fmul_rn(gamma, lv);      // buffers.py:88 (t == T-1); prescaled: fp16 bootstrap
        for (int j = 0; j < slices; ++j) {
            PipeStage &st = S.st[j % PG_STAGES];
            const int row0 = (slices - 1 - j) * PG_ROWS;
            const int rows = (int)(T - row0 < PG_ROWS ? T - row0 : PG_ROWS);
            const unsigned ph = (unsigned)(j / PG_STAGES) & 1u;
            mbar_wait(smem_u32(&S.full[j % PG_STAGES]), ph);
            const float gvn_next = __fmul_rn(gamma, st.v[0][lane]);         // for the slice before this one in time
            // delta[t] = (r[t] + (gamma * v[t+1]) * nnt[t]) - v[t] (buffers.py:88-90)
#pragma unroll
            for (int i = warp - 1; i < PG_ROWS; i += PG_DWARPS) {
                if (i < rows) {
                    const float gv = i + 1 < rows ? __fmul_rn(gamma, st.v[i + 1][lane]) : gvn;
                    const float nn = st.d[i][lane] ? 0.0f : 1.0f;
                    st.r[i][lane] = __fsub_rn(__fadd_rn(st.r[i][lane], __fmul_rn(gv, nn)), st.v[i][lane]);
                }
            }
            gvn = gvn_next;
            mbar_arrive(smem_u32(&S.dd[j % PG_STAGES]));
        }
        return;
    }

    // ---- walk warp: last = delta + ((gamma*lam) * nnt) * last (buffers.py:91) and returns = advantages + values
    // (buffers.py:94); rows beyond `rows` (the ragged newest slice) are skipped
    float last = 0.0f;                                          // buffers.py:86
    for (int j = 0; j < slices; ++j) {
        PipeStage &st = S.st[j % PG_STAGES];
        const int row0 = (slices - 1 - j) * PG_ROWS;
        const int rows = (int)(T - row0 < PG_ROWS ? T - row0 : PG_ROWS);
        const unsigned ph = (unsigned)(j / PG_STAGES) & 1u;
        mbar_wait(smem_u32(&S.dd[j % PG_STAGES]), ph);
        // BATCH rows of the column go to registers ahead of the dependent FMUL -> FADD chain.  BATCH = 32 (the whole
        // slice, 96 loads in flight, 127 registers): the chain never waits for shared memory -- 5.2 instead of 6.2-7.1 us
        // at T=128, N=8,192, where the walk is the critical path -- but only 3 CTAs fit an SM, which costs 9 % when
        // the kernel is bandwidth-bound; BATCH = 8 (40 registers, 5 CTAs per SM) is the shape for many columns.
        if (BATCH == PG_ROWS) {
            float dl[PG_ROWS], gl[PG_ROWS], vv[PG_ROWS];
#pragma unroll
            for (int i = 0; i < PG_ROWS; ++i) {
                dl[i] = st.r[i][lane];
                gl[i] = st.d[i][lane] ? 0.0f : gamma_lam;                   // == gamma_lam * nnt exactly
                vv[i] = st.v[i][lane];
            }
#pragma unroll
            for (int i = PG_ROWS - 1; i >= 0; --i) {
                if (i < rows) {
                    last = __fadd_rn(dl[i], __fmul_rn(gl[i], last));
                    st.r[i][lane] = last;
                    st.v[i][lane] = __fadd_rn(last, vv[i]);
                }
            }
        } else {
#pragma unroll
            for (int hi = PG_ROWS; hi > 0; hi -= BATCH) {
                float dl[BATCH], gl[BATCH], vv[BATCH];
#pragma unroll
                for (int q = 0; q < BATCH; ++q) {
                    dl[q] = st.r[hi - 1 - q][lane];
                    gl[q] = st.d[hi - 1 - q][lane] ? 0.0f : gamma_lam;      // == gamma_lam * nnt exactly
                    vv[q] = st.v[hi - 1 - q][lane];
                }
#pragma unroll
                for (int q = 0; q < BATCH; ++q) {
                    const int i = hi - 1 - q;
                    if (i < rows) {
                        last = __fadd_rn(dl[q], __fmul_rn(gl[q], last));
                        st.r[i][lane] = last;
                        st.v[i][lane] = __fadd_rn(last, vv[q]);
                    }
                }
            }
        }
        fence_proxy_async();                    // generic-proxy writes -> visible to the TMA store
        mbar_arrive(smem_u32(&S.done[j % PG_STAGES]));
    }
}

// [T][N] row-major array of `es`-byte elements, box = [PG_ROWS][PG_COLS]
static bool make_map(CUtensorMap *m, const void *base, CUtensorMapDataType dt, size_t es, int64_t T, int64_t N)
{
    const cuuint64_t dims[2] = {(cuuint64_t)N, (cuuint64_t)T};
    const cuuint64_t strides[1] = {(cuuint64_t)N * es};
    const cuuint32_t box[2] = {PG_COLS, PG_ROWS};
    return encode_tiled(m, dt, 2, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE) == CUDA_SUCCESS;
}

}  // namespace msw

extern "C" int msw_gae(const float *rewards, const float *values, const uint8_t *dones,
                       const float *last_values, float *advantages, float *returns, int64_t T,
                       int64_t N, float gamma_f32, float gamma_lam_f32, int32_t last_values_prescaled,
                       void *stream)
{
    using namespace msw;
    if (!rewards || !values || !dones || !last_values || !advantages || !returns)
        return fail(MSW_ERR_NULL, "msw_gae: NULL pointer");
    if (T < 0 || N < 0) return fail(MSW_ERR_BAD_SHAPE, "msw_gae: T=%lld N=%lld", (long long)T, (long long)N);
    if (T == 0 || N == 0) return MSW_OK;
    const long long blocks = (N + COLS - 1) / COLS;
    if (blocks > 0x7fffffffLL) return fail(MSW_ERR_BAD_SHAPE, "msw_gae: N too large");
    // TMA kernel where the tensor maps can be built (16-byte aligned bases and row pitches: N % 16 == 0, N bytes
    // for dones); the plain-load kernel serves ragged N.  One kernel per shape class, no run-time switch.
    const uintptr_t bases = (uintptr_t)rewards | (uintptr_t)values | (uintptr_t)dones | (uintptr_t)advantages | (uintptr_t)returns;
    if (N % 16 == 0 && (bases & 15u) == 0 && T <= 0x7fffffffLL && tensor_map_encoder_available()) {
        CUtensorMap mr, mv, md, ma, mt;
        if (!make_map(&mr, rewards, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, T, N) ||
            !make_map(&mv, values, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, T, N) ||
            !make_map(&md, dones, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, T, N) ||
            !make_map(&ma, advantages, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, T, N) ||
            !make_map(&mt, returns, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, T, N))
            return fail(MSW_ERR_ARG, "msw_gae: cuTensorMapEncodeTiled failed (T=%lld N=%lld)", (long long)T, (long long)N);
        // One wave of 3 CTAs per SM or less: latency-bound, the walk is the critical path -> the walk warp holds a
        // whole slice column in registers (127 registers, 3 CTAs per SM).  More CTAs: bandwidth-bound -> 8-row
        // batches (40 registers, 5 CTAs per SM); the register-heavy shape costs 9 % there (205 vs 186 us).
        if (blocks <= 3LL * sm_count()) {
            MSW_SET_MAX_SMEM(gae_pipe_kernel<PG_ROWS>, sizeof(PipeSmem));
            gae_pipe_kernel<PG_ROWS><<<(unsigned)blocks, PG_THREADS, sizeof(PipeSmem), (cudaStream_t)stream>>>(
                mr, mv, md, ma, mt, last_values, T, N, gamma_f32, gamma_lam_f32, (int)last_values_prescaled);
        } else {
            MSW_SET_MAX_SMEM(gae_pipe_kernel<8>, sizeof(PipeSmem));
            gae_pipe_kernel<8><<<(unsigned)blocks, PG_THREADS, sizeof(PipeSmem), (cudaStream_t)stream>>>(
                mr, mv, md, ma, mt, last_values, T, N, gamma_f32, gamma_lam_f32, (int)last_values_prescaled);
        }
        MSW_CUDA_TRY(cudaGetLastError());
        return MSW_OK;
    }
    gae_kernel<<<(unsigned)blocks, GAE_THREADS, 0, (cudaStream_t)stream>>>(
        rewards, values, dones, last_values, advantages, returns, T, N, gamma_f32, gamma_lam_f32, (int)last_values_prescaled);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}
