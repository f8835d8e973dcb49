// msw_env.cu -- vectorised Minesweeper environment kernels for sm_100a and
// their C-ABI entry points (include/msw_b200.h).
//
// One warp owns one board at a time (boards are independent: env.py:491-505
// touches only envs[i]).  The whole of VecMinesweeper.step -- action decode,
// first-click-safe mine placement, adjacency counts, flood-fill reveal, win /
// loss, reward, auto-reset, observation planes, action mask and the auxiliary
// mine label / valid maps -- is ONE kernel: the ~100 B of board state lives in
// registers between the step logic and the encoder, and the only HBM traffic
// that matters is the 10.5 KB (16x16) of fp32 observation + mask each warp
// streams out with 128-bit stores.  The kernel is HBM-write bound by design;
// the flood fill is latency-bound but hidden behind other warps' stores.
#include "../../include/msw_b200.h"
#include "msw_common.cuh"
#include "msw_error.h"

#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>


namespace msw {

// msw_host_expand.cpp: packed state -> the reference's fp32 observation planes / bool mask, on host threads
void expand_obs_host(int H, int W, const uint32_t *mines, const uint32_t *revealed, const int32_t *meta, long long n,
                     float *obs, uint8_t *mask, uint64_t *shadow, int shadow_valid, int threads);

struct EnvParams {
    int H, W, HW, wpb;
    int mine_count, safe;
    float r_step, r_loss, r_win;
    uint32_t k0, k1;                 // sampler key (seed)
    uint32_t thresh16;               // 65536 % HW (Lemire rejection threshold)
    long long env_id_base;
    long long n;
    // state
    uint32_t *mines, *revealed, *flags;
    int4 *meta;
    // step inputs
    const int32_t *a32;
    const long long *a64;
    const uint32_t *inj_bits;
    const uint8_t *inj_sel;
    // step outputs
    float *reward;
    uint8_t *done;
    int8_t *outcome;
    int32_t *new_reveals, *step, *rcount;
    // encode outputs
    float *obs;
    uint8_t *mask;
    float *labels;
    uint8_t *valid;
    // built-in synthetic policy (msw_step_io.rand_mode)
    int rand_mode;
    uint32_t rk0, rk1, rand_step;
    int32_t *a_out;
    int vec_mode;                    // 1: 4 cells / lane, 128-bit stores (HW % 4 == 0); 0: scalar
    // launch shape (launch_env): warps [0, wa) walk boards [0, na) with stride wa, warps [wa, wa + wb) walk
    // boards [na, nb) with stride wb, the remaining warps own one board each of [nb, n)
    long long seg_wa, seg_na, seg_wb, seg_nb;
    // per-lane geometry
    uint32_t g_valid[32], g_notcol0[32], g_notlast[32];
};

enum { MODE_STEP = 0, MODE_RESET = 1, MODE_ENCODE = 2 };

// ---------------------------------------------------------------------------
// First-click-safe placement (replaces env.py:280-312).  Forbidden set and the
// tiny-board fallback follow the reference; the subset itself is drawn with the
// counter-based sampler specified in DESIGN.md (NumPy's PCG64 stream is outside
// the parity contract).  Specification: a stream of 16-bit draws p = 0,1,2,...;
// draw p is 16-bit slot (p%256)/32 of Philox block 32*(p/256) + p%32 keyed by
// (seed; env id, episode); each draw proposes cell floor(x*HW/2^16) (Lemire,
// rejected when (x*HW mod 2^16) < 2^16 mod HW) and is accepted iff the cell is
// neither forbidden nor already chosen; stop at mine_count accepted cells
// (complement when more than half of the allowed cells are mines).  Sequential
// rejection sampling without replacement is exactly uniform over subsets.
//
// Evaluation is warp-parallel and order-exact: lane l owns Philox block
// 32*batch + l, so one round tests 32 consecutive draws at once; a draw is
// "novel" if its cell is free and no lower lane proposes the same cell
// (match.any), and only the first (K - accepted) novel draws are kept (ballot +
// lane-mask popcount), which is exactly what the sequential walk would do.
// ---------------------------------------------------------------------------
template <int CW, int CHW>
__device__ __noinline__ uint32_t sample_mines(const EnvParams &p, long long env_id, uint32_t episode,
                                              uint32_t startmask, int lane, const Geo &g)
{
    const int W = CW ? CW : p.W;
    const int HW = CHW ? CHW : p.HW;
    const int wpb = (HW + 31) >> 5;
    const int M = p.mine_count;
    uint32_t forb = startmask;
    if (p.safe) forb |= dilate8<CW>(startmask, lane, W, g);          // env.py:288-299
    int allowed = HW - warp_popc_sum(forb);
    if (allowed < M) {                                               // env.py:303-307
        forb = startmask;
        allowed = HW - 1;
    }
    const bool comp = 2 * M > allowed;          // sample the complement when dense
    const int K = comp ? allowed - M : M;
    const uint32_t thresh = CHW ? (65536u % (uint32_t)(CHW ? CHW : 1)) : p.thresh16;
    const uint32_t id_lo = (uint32_t)(unsigned long long)env_id;
    const uint32_t id_hi = (uint32_t)((unsigned long long)env_id >> 32);
    const uint32_t lt_mask = (1u << lane) - 1u;

    uint32_t chosen = 0;
    int cnt = 0;
    for (uint32_t batch = 0; cnt < K; ++batch) {
        uint32_t w[4];
        philox4x32_10(p.k0, p.k1, id_lo, id_hi, episode, batch * 32u + (uint32_t)lane, w);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            if (cnt >= K) break;
            const uint32_t x = (w[r >> 1] >> (16 * (r & 1))) & 0xFFFFu;
            const uint32_t m = x * (uint32_t)HW;
            const uint32_t d = m >> 16;
            const int owner = (int)(d >> 5);
            const uint32_t bit = 1u << (d & 31u);
            const uint32_t occ = __shfl_sync(FULL, forb | chosen, owner);
            const bool cand = ((m & 0xFFFFu) >= thresh) && !(occ & bit);
            const uint32_t same = __match_any_sync(FULL, cand ? d : (0x10000u + (uint32_t)lane));
            const bool novel = cand && ((same & lt_mask) == 0u);
            const uint32_t B = __ballot_sync(FULL, novel);
            const int need = K - cnt;
            const bool keep = novel && (__popc(B & lt_mask) < need);
            const int got = __popc(B);
            cnt += got < need ? got : need;
            for (int wd = 0; wd < wpb; ++wd) {
                const uint32_t nb = __reduce_or_sync(FULL, (keep && owner == wd) ? bit : 0u);
                if (lane == wd) chosen |= nb;
            }
        }
    }
    return comp ? (g.valid & ~forb & ~chosen) : chosen;
}

// ---------------------------------------------------------------------------
// Encoder: _build_obs (env.py:172-192), _compute_action_mask (env.py:194-196)
// and the aux maps of train_rl.py:205-212, from register-resident bitboards.
// Vector path (HW % 4 == 0): lane handles cells [4q, 4q+4) of every plane; the
// four {0,1} cells of a plane are a nibble that indexes a 16-entry float4 table
// in shared memory, so each 16-byte store costs two LOP3, one LDS.128 and one
// st.global.cs.v4.f32 (every warp store covers 512 contiguous bytes).
// ---------------------------------------------------------------------------
template <int CW, int CHW>
__device__ __forceinline__ void encode_board(const EnvParams &p, long long b, int lane, uint32_t R,
                                             uint32_t M, uint32_t F, int first, const Planes &pl,
                                             const Geo &g, const float4 *__restrict__ lut)
{
    const int HW = CHW ? CHW : p.HW;
    if (p.vec_mode == 1) {
        const int quads = HW >> 2;
        float4 *obs_b = p.obs ? reinterpret_cast<float4 *>(p.obs + b * (long long)(MSW_OBS_CHANNELS * HW)) : nullptr;
        uint32_t *mask_b = p.mask ? reinterpret_cast<uint32_t *>(p.mask + b * (long long)HW) : nullptr;
        float4 *lab_b = p.labels ? reinterpret_cast<float4 *>(p.labels + b * (long long)HW) : nullptr;
        uint32_t *val_b = p.valid ? reinterpret_cast<uint32_t *>(p.valid + b * (long long)HW) : nullptr;
        const uint32_t gate = first ? 15u : 0u;                       // env.py:181
#pragma unroll 2
        for (int q0 = 0; q0 < quads; q0 += 32) {
            const int q = q0 + lane;
            const bool act = q < quads;
            const int src = (act ? q : 0) >> 3;
            const int sh = (q & 7) << 2;
            const uint32_t r4 = (__shfl_sync(FULL, R, src) >> sh) & 15u;
            const uint32_t a0 = __shfl_sync(FULL, pl.c0, src) >> sh;
            const uint32_t a1 = __shfl_sync(FULL, pl.c1, src) >> sh;
            const uint32_t a2 = __shfl_sync(FULL, pl.c2, src) >> sh;
            const uint32_t a3 = __shfl_sync(FULL, pl.c3, src) >> sh;
            uint32_t l4 = 0, f4 = 0;
            if (lab_b) l4 = (__shfl_sync(FULL, M, src) >> sh) & gate;           // train_rl.py:206-208
            if (val_b && p.flags) f4 = (__shfl_sync(FULL, F, src) >> sh) & 15u;
            if (!act) continue;
            const uint32_t n4 = r4 ^ 15u;                                        // env.py:195
            if (obs_b) {
                const uint32_t g4 = r4 & gate;
                float4 *o = obs_b + q;
                __stcs(o, lut[r4]);
#pragma unroll
                for (int k = 0; k < 9; ++k) {
                    const uint32_t lo = g4 & ((k & 1) ? a0 : ~a0) & ((k & 2) ? a1 : ~a1);
                    const uint32_t m = lo & ((k & 4) ? a2 : ~a2) & ((k & 8) ? a3 : ~a3);
                    __stcs(o + (1 + k) * quads, lut[m]);
                }
            }
            if (mask_b) __stcs(mask_b + q, nib_to_b4(n4));
            if (lab_b) __stcs(lab_b + q, lut[l4]);
            if (val_b) __stcs(val_b + q, nib_to_b4(n4 & ~f4 & gate));            // train_rl.py:209
        }
    } else {
        // Scalar path for boards whose planes are not 16-byte multiples (e.g. 5x7, 9x9).
        const uint32_t Lm = first ? M : 0u;
        const uint32_t Vm = first ? (~R & ~F & g.valid) : 0u;
        const int wpb = (HW + 31) >> 5;
        float *obs_b = p.obs ? p.obs + b * (long long)(MSW_OBS_CHANNELS * HW) : nullptr;
        uint8_t *mask_b = p.mask ? p.mask + b * (long long)HW : nullptr;
        float *lab_b = p.labels ? p.labels + b * (long long)HW : nullptr;
        uint8_t *val_b = p.valid ? p.valid + b * (long long)HW : nullptr;
        for (int it = 0; it < wpb; ++it) {
            const int cell = it * 32 + lane;
            const uint32_t r = (__shfl_sync(FULL, R, it) >> lane) & 1u;
            const uint32_t cnt = ((__shfl_sync(FULL, pl.c0, it) >> lane) & 1u) |
                                 (((__shfl_sync(FULL, pl.c1, it) >> lane) & 1u) << 1) |
                                 (((__shfl_sync(FULL, pl.c2, it) >> lane) & 1u) << 2) |
                                 (((__shfl_sync(FULL, pl.c3, it) >> lane) & 1u) << 3);
            const uint32_t l = (__shfl_sync(FULL, Lm, it) >> lane) & 1u;
            const uint32_t v = (__shfl_sync(FULL, Vm, it) >> lane) & 1u;
            if (cell >= HW) continue;
            if (obs_b) {
                obs_b[cell] = r ? 1.0f : 0.0f;
                for (int k = 0; k < 9; ++k)
                    obs_b[(1 + k) * HW + cell] = (first && r && cnt == (uint32_t)k) ? 1.0f : 0.0f;
            }
            if (mask_b) mask_b[cell] = (uint8_t)(r ^ 1u);
            if (lab_b) lab_b[cell] = l ? 1.0f : 0.0f;
            if (val_b) val_b[cell] = (uint8_t)v;
        }
    }
}

// Lemire's multiply-shift with rejection over the four words of one Philox block (shared by the
// standalone action source and the built-in synthetic policy so both draw the same actions).
__device__ __forceinline__ uint32_t bounded(const uint32_t (&w)[4], uint32_t range)
{
    const uint32_t thresh = (0u - range) % range;
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const unsigned long long m = (unsigned long long)w[i] * range;
        r = (uint32_t)(m >> 32);
        if ((uint32_t)m >= thresh) break;
    }
    return r;
}


// Uniformly random unrevealed cell (or any cell) of the board held in R, warp-parallel; identical
// to random_actions_kernel for the same (seed, env id, step).
__device__ __forceinline__ int synth_action(const EnvParams &p, long long b, uint32_t R, int lane, int HW, const Geo &g)
{
    const unsigned long long id = (unsigned long long)(p.env_id_base + b);
    uint32_t w[4];
    philox4x32_10(p.rk0, p.rk1 ^ 0x41435431u, (uint32_t)id, (uint32_t)(id >> 32), p.rand_step, 0x5eedac71u, w);
    if (p.rand_mode != 1) return (int)bounded(w, (uint32_t)HW);
    const uint32_t free_cells = ~R & g.valid;
    const int c = __popc(free_cells);
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
    }
    const int total = __shfl_sync(FULL, incl, 31);
    if (total == 0) return 0;
    const int k = (int)bounded(w, (uint32_t)total);
    const unsigned over = __ballot_sync(FULL, incl > k);
    const int owner = __ffs(over) - 1;
    int a = 0;
    if (lane == owner) a = lane * 32 + (int)__fns(free_cells, 0, k - (incl - c) + 1);
    return __shfl_sync(FULL, a, owner);
}

// ---------------------------------------------------------------------------
// The fused env kernel.  MODE_STEP: VecMinesweeper.step (env.py:479-511);
// MODE_RESET: VecMinesweeper.reset (env.py:468-477); MODE_ENCODE: observation
// of the current state.  CW/CHW != 0 specialise the board shape at compile time.
// Each warp walks boards b, b+total_warps, ... and issues the loads of its next
// board before it starts computing on the current one, so the ~1 us of HBM/L2
// latency on the state is hidden behind the step logic and the stores.
// ---------------------------------------------------------------------------
struct BoardIn {
    uint32_t M, R, F;
    int4 meta;                 // first_click_done, step_count, episode_idx, last_new_reveals
    int a_lo, a_hi;            // raw action words; decoded at use so the prefetch never waits
};

template <int MODE>
__device__ __forceinline__ BoardIn load_board(const EnvParams &p, long long b, int lane, int wpb, uint64_t keep)
{
    BoardIn in;
    in.M = in.R = in.F = 0u;
    in.a_lo = in.a_hi = 0;
    in.meta = ld_keep(p.meta + b, keep);
    if (MODE != MODE_RESET && lane < wpb) {
        in.M = ld_keep(p.mines + b * wpb + lane, keep);
        in.R = ld_keep(p.revealed + b * wpb + lane, keep);
        if (p.flags) in.F = ld_keep(p.flags + b * wpb + lane, keep);
    }
    if (MODE == MODE_STEP && !p.rand_mode) {
        if (p.a32) {
            in.a_lo = __ldg(p.a32 + b);
        } else {
            const int2 a = __ldg(reinterpret_cast<const int2 *>(p.a64) + b);
            in.a_lo = a.x;
            in.a_hi = a.y;
        }
    }
    return in;
}

template <int MODE, int CW, int CHW, bool PF, int MINB>
__global__ void __launch_bounds__(256, MINB) env_kernel(const __grid_constant__ EnvParams p)
{
    __shared__ float4 s_lut[16];                 // nibble of four {0,1} cells -> four fp32
    if (threadIdx.x < 16) s_lut[threadIdx.x] = nib_to_f4(threadIdx.x);
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int W = CW ? CW : p.W;
    const int HW = CHW ? CHW : p.HW;
    const int wpb = (HW + 31) >> 5;
    const long long warps_per_block = blockDim.x >> 5;
    Geo g;
    g.valid = p.g_valid[lane];
    g.notcol0 = p.g_notcol0[lane];
    g.notlast = p.g_notlast[lane];
    const bool own = lane < wpb;
    const uint64_t keep = l2_keep_policy();

    // Which boards this warp walks: b, b + stride, ... below `end` (three segments, see launch_env: late CTAs get
    // fewer boards so that the grid drains over one board time instead of three)
    const long long w = (long long)blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    long long b, end;
    int stride;                                          // a segment never has more than 2^31 warps (grid limit)
    if (w < p.seg_wa) {
        b = w; stride = (int)p.seg_wa; end = p.seg_na;
    } else if (w < p.seg_wa + p.seg_wb) {
        b = p.seg_na + (w - p.seg_wa); stride = (int)p.seg_wb; end = p.seg_nb;
    } else {
        b = p.seg_nb + (w - p.seg_wa - p.seg_wb); stride = 1; end = b + 1 < p.n ? b + 1 : p.n;
    }
    if (b >= end) return;
    int left = (int)((end - b + stride - 1) / stride);   // boards this warp walks (once per warp; keeps `end` out of the loop)
    BoardIn cur = load_board<MODE>(p, b, lane, wpb, keep);
    while (true) {
        const long long nb = b + stride;
        const bool more = --left > 0;
        BoardIn nxt;
        if (PF && more) nxt = load_board<MODE>(p, nb, lane, wpb, keep);   // prefetch: consumed next iteration

        uint32_t M = cur.M, R = cur.R, F = cur.F;
        const int4 meta = cur.meta;
        int first = meta.x;
        Planes pl = {0u, 0u, 0u, 0u};

        if (MODE == MODE_RESET) {
            // env.py:87-95: zero everything; the sampler counter moves on (the reference's
            // per-env Generator is never re-seeded either, env.py:49).
            first = 0;
            if (own) {
                st_keep(p.mines + b * wpb + lane, 0u, keep);
                st_keep(p.revealed + b * wpb + lane, 0u, keep);
                if (p.flags) st_keep(p.flags + b * wpb + lane, 0u, keep);
            }
            if (lane == 0) st_keep(p.meta + b, make_int4(0, 0, meta.z + 1, 0), keep);
        } else if (MODE == MODE_ENCODE) {
            if (first) pl = count_planes<CW>(M, lane, W, g);
        } else {
            // ---- action decode: cell = action % (H*W), Python modulo (env.py:104-107)
            int cell;
            if (p.rand_mode) {
                cell = synth_action(p, b, R, lane, HW, g);
                if (p.a_out && lane == 0) p.a_out[b] = cell;
            } else if (p.a32 || cur.a_hi == (cur.a_lo >> 31)) {
                cell = cur.a_lo % HW;                                     // fits int32
            } else {
                const long long a = ((long long)cur.a_hi << 32) | (unsigned int)cur.a_lo;
                cell = (int)(a % (long long)HW);
            }
            if (cell < 0) cell += HW;
            const uint32_t startmask = (lane == (cell >> 5)) ? (1u << (cell & 31)) : 0u;

            int done = 0, outcome = 0, newly = 0;
            bool mines_dirty = false, reveal_branch = false;
            if (!__any_sync(FULL, R & startmask)) {                       // env.py:118
                if (!first) {                                             // env.py:119-122
                    if (p.inj_sel && p.inj_sel[b])
                        M = own ? (p.inj_bits[b * wpb + lane] & g.valid) : 0u;
                    else
                        M = sample_mines<CW, CHW>(p, p.env_id_base + b, (uint32_t)meta.z, startmask, lane, g);
                    first = 1;
                    mines_dirty = true;
                }
                pl = count_planes<CW>(M, lane, W, g);                     // env.py:314-335
                if (__any_sync(FULL, M & startmask)) {                    // env.py:124-128
                    R |= startmask;
                    done = 1;
                    outcome = 2;
                } else {                                                  // env.py:129-133
                    // Flood fill (env_numba.py:16-77) as a least fixed point: S grows by the
                    // 8-neighbours of its zero-count cells that are not revealed / flagged /
                    // mines; only the newest zero cells (the frontier) need dilating.
                    const uint32_t zero = ~(pl.c0 | pl.c1 | pl.c2 | pl.c3) & g.valid;
                    const uint32_t blocked = R | F | M;
                    uint32_t S = startmask & ~F;                          // env.py:200 guard
                    uint32_t front = S & zero;
                    while (__any_sync(FULL, front)) {
                        const uint32_t D = dilate8<CW>(front, lane, W, g) & ~blocked & ~S;
                        S |= D;
                        front = D & zero;
                    }
                    newly = warp_popc_sum(S);
                    R |= S;
                    reveal_branch = true;
                }
            } else if (first) {
                pl = count_planes<CW>(M, lane, W, g);                     // no-op click, env.py:138-140
            }
            const int total = warp_popc_sum(R);
            if (reveal_branch && total >= HW - p.mine_count) {            // env.py:134-137
                done = 1;
                outcome = 1;
            }
            const int step_now = meta.y + 1;                              // env.py:143

            if (lane == 0) {                                              // env.py:493-505
                p.reward[b] = done ? (outcome == 1 ? p.r_win : p.r_loss) : p.r_step;
                p.done[b] = (uint8_t)done;
                if (p.outcome) p.outcome[b] = (int8_t)outcome;
                if (p.new_reveals) p.new_reveals[b] = newly;
                if (p.step) p.step[b] = step_now;
                if (p.rcount) p.rcount[b] = total;
            }
            if (done) {                                                   // auto-reset, env.py:497-498
                M = 0u; R = 0u; F = 0u;
                first = 0;
                pl.c0 = pl.c1 = pl.c2 = pl.c3 = 0u;
                if (own && p.flags) st_keep(p.flags + b * wpb + lane, 0u, keep);
                if (lane == 0) st_keep(p.meta + b, make_int4(0, 0, meta.z + 1, 0), keep);
            } else if (lane == 0) {
                st_keep(p.meta + b, make_int4(first, step_now, meta.z, newly), keep);
            }
            if (own) {
                st_keep(p.revealed + b * wpb + lane, R, keep);
                if (mines_dirty || done) st_keep(p.mines + b * wpb + lane, M, keep);
            }
        }
        encode_board<CW, CHW>(p, b, lane, R, M, F, first, pl, g, s_lut);
        if (!more) break;
        if (PF) cur = nxt;
        else cur = load_board<MODE>(p, nb, lane, wpb, keep);
        b = nb;
    }
}

// ---------------------------------------------------------------------------
// Late-start curriculum (env.py:416-466; SURVEY section 8 row f3), applied to freshly reset boards:
// with probability `prob` pre-play random SAFE cells until at most `target_hidden` safe cells stay
// hidden.  Control flow follows the reference line by line; randomness comes from a counter-based
// stream (the reference shares ONE sequential NumPy generator over all envs, env.py:397-403, which
// no parallel implementation can reproduce): draw k of env e is word k%4 of Philox block k/4, key =
// late-start seed, counter = (env id lo, env id hi, episode index at entry, block); DESIGN.md
// section 2 specifies the stream, the test-side restatement follows the same specification.
// ---------------------------------------------------------------------------
struct LateParams {
    EnvParams e;
    const uint8_t *sel;          // nullable [n]: apply only where sel != 0 (the envs a step just reset)
    uint32_t lk0, lk1;           // late-start seed
    uint32_t prob24;             // prob * 2^24
    int min_hidden, max_hidden, max_attempts, max_extra_steps;
};

struct LateRng {
    uint32_t k0, k1, c0, c1, c2, idx;
    uint32_t w[4];
    __device__ __forceinline__ uint32_t next()
    {
        if ((idx & 3u) == 0u) philox4x32_10(k0, k1, c0, c1, c2, idx >> 2, w);
        const uint32_t i = idx & 3u;
        ++idx;
        return i == 0 ? w[0] : i == 1 ? w[1] : i == 2 ? w[2] : w[3];
    }
    // Lemire bounded integer with rejection (fresh words on rejection)
    __device__ __forceinline__ uint32_t below(uint32_t range)
    {
        const uint32_t thresh = (0u - range) % range;
        while (true) {
            const unsigned long long m = (unsigned long long)next() * range;
            if ((uint32_t)m >= thresh) return (uint32_t)(m >> 32);
        }
    }
};

__global__ void __launch_bounds__(128) late_start_kernel(const __grid_constant__ LateParams q)
{
    const EnvParams &p = q.e;
    const int lane = threadIdx.x & 31;
    const int W = p.W, HW = p.HW, wpb = p.wpb;
    const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= p.n) return;
    if (q.sel && !q.sel[b]) return;
    Geo g;
    g.valid = p.g_valid[lane];
    g.notcol0 = p.g_notcol0[lane];
    g.notlast = p.g_notlast[lane];
    const bool own = lane < wpb;
    int4 meta = p.meta[b];
    uint32_t M = 0, R = 0, F = 0;
    if (own) {
        M = p.mines[b * wpb + lane];
        R = p.revealed[b * wpb + lane];
        if (p.flags) F = p.flags[b * wpb + lane];
    }
    int first = meta.x, step_count = meta.y, last_new = meta.w;
    uint32_t episode = (uint32_t)meta.z;
    const unsigned long long id = (unsigned long long)(p.env_id_base + b);
    LateRng rng = {q.lk0, q.lk1, (uint32_t)id, (uint32_t)(id >> 32), episode, 0u, {0u, 0u, 0u, 0u}};

    if ((rng.next() >> 8) >= q.prob24) return;                       // rng.random() >= prob (env.py:422)
    const int safe_total = HW - p.mine_count;
    Planes pl = {0u, 0u, 0u, 0u};
    if (first) pl = count_planes<0>(M, lane, W, g);

    // MinesweeperEnv.step on a cell known to be unrevealed and (after placement) not a mine
    auto click = [&](int cell) -> bool {
        const uint32_t startmask = (lane == (cell >> 5)) ? (1u << (cell & 31)) : 0u;
        if (!first) {
            M = sample_mines<0, 0>(p, p.env_id_base + b, episode, startmask, lane, g);
            first = 1;
            pl = count_planes<0>(M, lane, W, g);
        }
        const uint32_t zero = ~(pl.c0 | pl.c1 | pl.c2 | pl.c3) & g.valid;
        const uint32_t blocked = R | F | M;
        uint32_t S = startmask & ~F;
        uint32_t front = S & zero;
        while (__any_sync(FULL, front)) {
            const uint32_t D = dilate8<0>(front, lane, W, g) & ~blocked & ~S;
            S |= D;
            front = D & zero;
        }
        last_new = warp_popc_sum(S);
        R |= S;
        step_count += 1;
        return warp_popc_sum(R) >= safe_total;                        // win (env.py:134-137)
    };
    auto fresh = [&]() {                                              // env.reset(), env.py:87-95
        M = 0u; R = 0u; F = 0u;
        first = 0; step_count = 0; last_new = 0;
        episode += 1u;
        pl.c0 = pl.c1 = pl.c2 = pl.c3 = 0u;
    };

    bool success = false;
    for (int attempt = 0; attempt < q.max_attempts && !success; ++attempt) {
        if (first) fresh();                                           // env.py:437-438
        bool done = click((int)rng.below((uint32_t)HW));              // env.py:441-442
        if (done) continue;
        int target = q.min_hidden + (int)rng.below((uint32_t)(q.max_hidden - q.min_hidden + 1));   // :446
        target = target < 1 ? 1 : (target > safe_total ? safe_total : target);                     // :447
        for (int e = 0; e < q.max_extra_steps; ++e) {                 // env.py:449-458
            if (safe_total - warp_popc_sum(R) <= target) { success = true; break; }
            const uint32_t cand = ~M & ~R & ~F & g.valid;
            const int c = __popc(cand);
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += t;
            }
            const int total = __shfl_sync(FULL, incl, 31);
            if (total == 0) break;
            const int k = (int)rng.below((uint32_t)total);           // rng.choice(safe_candidates)
            const int owner = __ffs(__ballot_sync(FULL, incl > k)) - 1;
            int cell = 0;
            if (lane == owner) cell = lane * 32 + (int)__fns(cand, 0, k - (incl - c) + 1);
            cell = __shfl_sync(FULL, cell, owner);
            done = click(cell);
            if (done) break;
        }
        if (!success && !done && safe_total - warp_popc_sum(R) <= target) success = true;   // env.py:460-462
    }
    if (!success) fresh();                                            // env.py:465-466
    if (own) {
        p.mines[b * wpb + lane] = M;
        p.revealed[b * wpb + lane] = R;
        if (p.flags) p.flags[b * wpb + lane] = F;
    }
    if (lane == 0) p.meta[b] = make_int4(first, step_count, (int)episode, last_new);
}

// ---------------------------------------------------------------------------
// Compact replay (SURVEY section 8 row f2): a transition is stored as the bitboards that generated
// its observation (mines + revealed [+ flags] + first_click_done: 65 B at 16x16 instead of the
// 11.8 KB of obs + mask + aux maps), and RolloutBuffer.get_minibatches' randperm gather
// (buffers.py:96-116) becomes this kernel: row j of the minibatch is re-encoded from snapshot
// idx[j] straight into the minibatch tensors.  Same encoder as the step kernel, so the result is
// bit-identical to gathering rows of a dense buffer.
// ---------------------------------------------------------------------------
struct GatherParams {
    EnvParams e;                     // geometry + destination pointers (obs/mask/labels/valid), n = rows out
    const uint32_t *s_mines, *s_revealed, *s_flags;   // [rows_in][wpb] (s_flags nullable)
    const uint8_t *s_first;          // [rows_in]
    const long long *idx;            // [n] source row of each output row
    long long rows_in;
};

template <int CW, int CHW>
__global__ void __launch_bounds__(256) gather_encode_kernel(const __grid_constant__ GatherParams q)
{
    __shared__ float4 s_lut[16];
    if (threadIdx.x < 16) s_lut[threadIdx.x] = nib_to_f4(threadIdx.x);
    __syncthreads();
    const EnvParams &p = q.e;
    const int lane = threadIdx.x & 31;
    const int W = CW ? CW : p.W;
    const int HW = CHW ? CHW : p.HW;
    const int wpb = (HW + 31) >> 5;
    const long long warps_per_block = blockDim.x >> 5;
    const long long total_warps = (long long)gridDim.x * warps_per_block;
    Geo g;
    g.valid = p.g_valid[lane];
    g.notcol0 = p.g_notcol0[lane];
    g.notlast = p.g_notlast[lane];
    for (long long j = (long long)blockIdx.x * warps_per_block + (threadIdx.x >> 5); j < p.n; j += total_warps) {
        long long src = q.idx[j];
        if (src < 0 || src >= q.rows_in) src = 0;               // host validates; never fault on a bad index
        uint32_t M = 0, R = 0, F = 0;
        if (lane < wpb) {
            M = __ldg(q.s_mines + src * wpb + lane);
            R = __ldg(q.s_revealed + src * wpb + lane);
            if (q.s_flags) F = __ldg(q.s_flags + src * wpb + lane);
        }
        const int first = q.s_first[src] != 0;
        Planes pl = {0u, 0u, 0u, 0u};
        if (first) pl = count_planes<CW>(M, lane, W, g);
        encode_board<CW, CHW>(p, j, lane, R, M, F, first, pl, g, s_lut);
    }
}

// ---------------------------------------------------------------------------
// Eval-side analytics (SURVEY section 8 row f4): rules.analyze_forced_modules (rules.py:206-259),
// the pairwise subset rule on ground-truth mines.  For number cells a, b (revealed, count > 0) with
// non-empty unknown-neighbour sets U(a), U(b) (unknown = not revealed; flags are ignored, :218):
// if U(a) is a subset of U(b) and both contain the same number of mines, every cell of U(b) - U(a) is
// safe.  A non-empty U(a) inside U(b) forces a and b within Chebyshev distance 2, so each number cell
// only needs its 5x5 window instead of the reference's all-pairs loop.  One warp per board; the three
// cell predicates are expanded to bytes in shared memory and each lane walks its cells with scalar
// code (this runs at eval batch sizes; clarity over speed).
// ---------------------------------------------------------------------------
struct SubsetParams {
    EnvParams e;
    uint32_t *out;      // [n][wpb] bitboard of "subset_reveal" cells
};

__global__ void __launch_bounds__(128) subset_reveal_kernel(const __grid_constant__ SubsetParams q)
{
    extern __shared__ unsigned char s_raw[];
    const EnvParams &p = q.e;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int H = p.H, W = p.W, HW = p.HW, wpb = p.wpb;
    const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    unsigned char *s_unknown = s_raw + (size_t)warp * (3 * MSW_MAX_CELLS + 128);
    unsigned char *s_mine = s_unknown + MSW_MAX_CELLS;
    unsigned char *s_number = s_mine + MSW_MAX_CELLS;
    uint32_t *s_res = reinterpret_cast<uint32_t *>(s_number + MSW_MAX_CELLS);
    if (b >= p.n) return;
    Geo g;
    g.valid = p.g_valid[lane];
    g.notcol0 = p.g_notcol0[lane];
    g.notlast = p.g_notlast[lane];
    uint32_t M = 0, R = 0;
    if (lane < wpb) {
        M = p.mines[b * wpb + lane];
        R = p.revealed[b * wpb + lane];
    }
    const Planes pl = count_planes<0>(M, lane, W, g);
    const uint32_t number = R & (pl.c0 | pl.c1 | pl.c2 | pl.c3) & g.valid;       // revealed & counts > 0 (:222)
    const uint32_t unknown = ~R & g.valid;                                        // :218
    for (int it = 0; it < wpb; ++it) {
        const int cell = it * 32 + lane;
        const uint32_t wu = __shfl_sync(FULL, unknown, it), wm = __shfl_sync(FULL, M, it), wn = __shfl_sync(FULL, number, it);
        if (cell < HW) {
            s_unknown[cell] = (wu >> lane) & 1u;
            s_mine[cell] = (wm >> lane) & 1u;
            s_number[cell] = (wn >> lane) & 1u;
        }
    }
    s_res[lane] = 0u;
    __syncwarp();

    // unknown neighbours of (r, c): fills idx[] and returns the count; *mines = mines among them
    auto unknown_nbrs = [&](int r, int c, int (&idx)[8], int *mines) {
        int k = 0, m = 0;
        for (int dr = -1; dr <= 1; ++dr)
            for (int dc = -1; dc <= 1; ++dc) {
                if (!dr && !dc) continue;
                const int rr = r + dr, cc = c + dc;
                if (rr < 0 || rr >= H || cc < 0 || cc >= W) continue;
                const int u = rr * W + cc;
                if (s_unknown[u]) {
                    idx[k++] = u;
                    m += s_mine[u];
                }
            }
        *mines = m;
        return k;
    };
    for (int a = lane; a < HW; a += 32) {
        if (!s_number[a]) continue;
        const int ra = a / W, ca = a % W;
        int ua[8], ma;
        const int na = unknown_nbrs(ra, ca, ua, &ma);
        if (na == 0) continue;                                                    // :230-231
        for (int br = -2; br <= 2; ++br)
            for (int bc = -2; bc <= 2; ++bc) {
                if (!br && !bc) continue;
                const int rb = ra + br, cb = ca + bc;
                if (rb < 0 || rb >= H || cb < 0 || cb >= W) continue;
                const int bb = rb * W + cb;
                if (!s_number[bb]) continue;
                int ub[8], mb;
                const int nb = unknown_nbrs(rb, cb, ub, &mb);
                if (nb == 0 || ma != mb) continue;                                // :251, :255
                bool subset = true;                                               // U(a) subset of U(b)?
                for (int k = 0; k < na && subset; ++k) {
                    const int dr = ua[k] / W - rb, dc = ua[k] % W - cb;
                    subset = dr >= -1 && dr <= 1 && dc >= -1 && dc <= 1;
                }
                if (!subset) continue;
                for (int k = 0; k < nb; ++k) {                                    // U(b) - U(a) is safe (:250-252)
                    const int dr = ub[k] / W - ra, dc = ub[k] % W - ca;
                    if (!(dr >= -1 && dr <= 1 && dc >= -1 && dc <= 1))
                        atomicOr(&s_res[ub[k] >> 5], 1u << (ub[k] & 31));
                }
            }
    }
    __syncwarp();
    if (lane < wpb) q.out[b * wpb + lane] = s_res[lane];
}

// Expansion of the bitboards into the reference's per-cell arrays for the
// vec.envs[i] views (env.py:68-71, adjacent_counts per env.py:314-335).
struct UnpackParams {
    EnvParams e;
    uint8_t *o_mine, *o_rev, *o_flags, *o_counts;
};

__global__ void __launch_bounds__(256) unpack_kernel(const __grid_constant__ UnpackParams q)
{
    const EnvParams &p = q.e;
    const int lane = threadIdx.x & 31;
    const int HW = p.HW, wpb = p.wpb;
    const long long warps_per_block = blockDim.x >> 5;
    const long long total_warps = (long long)gridDim.x * warps_per_block;
    Geo g;
    g.valid = p.g_valid[lane];
    g.notcol0 = p.g_notcol0[lane];
    g.notlast = p.g_notlast[lane];
    for (long long b = (long long)blockIdx.x * warps_per_block + (threadIdx.x >> 5); b < p.n; b += total_warps) {
        uint32_t M = 0, R = 0, F = 0;
        if (lane < wpb) {
            M = p.mines[b * wpb + lane];
            R = p.revealed[b * wpb + lane];
            if (p.flags) F = p.flags[b * wpb + lane];
        }
        const Planes pl = count_planes<0>(M, lane, p.W, g);
        for (int it = 0; it < wpb; ++it) {
            const int cell = it * 32 + lane;
            const uint32_t m = (__shfl_sync(FULL, M, it) >> lane) & 1u;
            const uint32_t r = (__shfl_sync(FULL, R, it) >> lane) & 1u;
            const uint32_t f = (__shfl_sync(FULL, F, it) >> lane) & 1u;
            const uint32_t cnt = ((__shfl_sync(FULL, pl.c0, it) >> lane) & 1u) |
                                 (((__shfl_sync(FULL, pl.c1, it) >> lane) & 1u) << 1) |
                                 (((__shfl_sync(FULL, pl.c2, it) >> lane) & 1u) << 2) |
                                 (((__shfl_sync(FULL, pl.c3, it) >> lane) & 1u) << 3);
            if (cell >= HW) continue;
            const long long o = b * (long long)HW + cell;
            if (q.o_mine) q.o_mine[o] = (uint8_t)m;
            if (q.o_rev) q.o_rev[o] = (uint8_t)r;
            if (q.o_flags) q.o_flags[o] = (uint8_t)f;
            if (q.o_counts) q.o_counts[o] = (uint8_t)cnt;
        }
    }
}

// Synthetic action source (BASELINE.md section 4): one thread per env.
struct ActParams {
    const uint32_t *revealed;
    int HW, wpb;
    long long n, env_id_base;
    uint32_t k0, k1, step_index;
    int valid_only;
    int32_t *a32;
    long long *a64;
};

__global__ void __launch_bounds__(256) random_actions_kernel(const ActParams p)
{
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.n) return;
    const unsigned long long id = (unsigned long long)(p.env_id_base + b);
    uint32_t w[4];
    philox4x32_10(p.k0, p.k1 ^ 0x41435431u, (uint32_t)id, (uint32_t)(id >> 32), p.step_index, 0x5eedac71u, w);
    int action = 0;
    if (!p.valid_only) {
        action = (int)bounded(w, (uint32_t)p.HW);
    } else {
        const uint32_t *R = p.revealed + b * p.wpb;
        int cnt = 0;
        for (int i = 0; i < p.wpb; ++i) {
            uint32_t valid = (i == p.wpb - 1 && (p.HW & 31)) ? ((1u << (p.HW & 31)) - 1u) : 0xffffffffu;
            cnt += __popc(~R[i] & valid);
        }
        if (cnt > 0) {
            int k = (int)bounded(w, (uint32_t)cnt);
            for (int i = 0; i < p.wpb; ++i) {
                uint32_t valid = (i == p.wpb - 1 && (p.HW & 31)) ? ((1u << (p.HW & 31)) - 1u) : 0xffffffffu;
                const uint32_t free_cells = ~R[i] & valid;
                const int c = __popc(free_cells);
                if (k < c) {
                    action = i * 32 + (int)__fns(free_cells, 0, k + 1);
                    break;
                }
                k -= c;
            }
        }
    }
    if (p.a32) p.a32[b] = action;
    if (p.a64) p.a64[b] = action;
}

// ---------------------------------------------------------------------------
// Host side of the C ABI
// ---------------------------------------------------------------------------
// Board geometry and env constants (no state pointers).
static int fill_geometry(EnvParams &p, const msw_env_desc *d, long long n)
{
    if (!d) return fail(MSW_ERR_NULL, "desc is NULL");
    if (d->H < 1 || d->W < 1 || d->W > 32 || (long long)d->H * d->W > MSW_MAX_CELLS)
        return fail(MSW_ERR_BAD_SHAPE, "board %dx%d unsupported (need 1<=W<=32, H*W<=%d)", d->H, d->W, MSW_MAX_CELLS);
    if (d->mine_count < 0 || d->mine_count > d->H * d->W - 1)
        return fail(MSW_ERR_BAD_SHAPE, "mine_count %d out of range for %dx%d", d->mine_count, d->H, d->W);
    if (n < 0) return fail(MSW_ERR_BAD_SHAPE, "n=%lld < 0", n);
    memset(&p, 0, sizeof(p));
    p.H = d->H; p.W = d->W; p.HW = d->H * d->W; p.wpb = (p.HW + 31) / 32;
    p.mine_count = d->mine_count; p.safe = d->safe_nbhd != 0;
    p.r_step = d->reward_step; p.r_loss = d->reward_loss; p.r_win = d->reward_win;
    p.k0 = (uint32_t)d->seed; p.k1 = (uint32_t)(d->seed >> 32);
    p.thresh16 = 65536u % (uint32_t)p.HW;
    p.env_id_base = d->env_id_base;
    p.n = n;
    for (int w = 0; w < 32; ++w) {
        uint32_t v = 0, a = 0, z = 0;
        for (int j = 0; j < 32; ++j) {
            const int cell = w * 32 + j;
            if (cell >= p.HW) break;
            const int col = cell % p.W;
            v |= 1u << j;
            if (col != 0) a |= 1u << j;
            if (col != p.W - 1) z |= 1u << j;
        }
        p.g_valid[w] = v; p.g_notcol0[w] = a; p.g_notlast[w] = z;
    }
    return MSW_OK;
}

// Geometry + the persistent env state.
static int fill_params(EnvParams &p, const msw_env_desc *d, const msw_state *st, long long n)
{
    if (!st) return fail(MSW_ERR_NULL, "state is NULL");
    if (!st->mines || !st->revealed || !st->meta) return fail(MSW_ERR_NULL, "state pointer is NULL");
    if (((uintptr_t)st->meta & 15u) != 0) return fail(MSW_ERR_ALIGN, "state.meta must be 16-byte aligned");
    const int rc = fill_geometry(p, d, n);
    if (rc) return rc;
    p.mines = st->mines; p.revealed = st->revealed; p.flags = st->flags;
    p.meta = reinterpret_cast<int4 *>(st->meta);
    return MSW_OK;
}

static int set_encode_out(EnvParams &p, const msw_encode_out *out, bool require)
{
    if (!out) return require ? fail(MSW_ERR_NULL, "encode outputs are NULL") : MSW_OK;
    p.obs = out->obs; p.mask = out->mask; p.labels = out->mine_labels; p.valid = out->mine_valid;
    const uintptr_t f = (uintptr_t)p.obs | (uintptr_t)p.labels, m = (uintptr_t)p.mask | (uintptr_t)p.valid;
    p.vec_mode = 0;
    if ((p.HW & 3) == 0) {
        if ((f & 15u) || (m & 3u))
            return fail(MSW_ERR_ALIGN, "obs/mine_labels must be 16-byte and mask/mine_valid 4-byte aligned");
        // (8 cells / lane with 256-bit st.global.v8 stores was measured 8% SLOWER than this
        // 128-bit path on B200 -- profiles/r01_sweep_vec256.txt -- and was removed.)
        p.vec_mode = 1;
    }
    return MSW_OK;
}

// Launch shape.  Stores reach full HBM write bandwidth only when CTAs are handed out
// dynamically (profiles/r01_store_probe2.txt: a static one-wave grid tops out near 6.0 TB/s,
// the same stores from many short CTAs reach 6.9-7.0 TB/s), so the grid is sized from
// boards-per-warp rather than from the SM count:
//   CTA = one warp (a slow board -- a deep flood fill, a board draw -- never holds other warps' slots),
//   3 boards per warp with the next board's state prefetched (80 registers).
// Sweeps: profiles/r01_sweep_launch_shape.txt, profiles/r01_sweep_*.txt, profiles/r02ao_bpw_taper_sweep.txt.
constexpr int ENV_BPW = 3;

// Fills the three launch segments of `q` and returns the grid of one-warp CTAs.  Most warps walk 3 boards (next board's state
// prefetched); CTAs are handed out in index order, so the LAST CTAs get two boards, then one: when the grid runs
// out of CTAs the SMs otherwise drain over a whole 3-board CTA lifetime (~18 us of a 110 us launch at C2) with
// falling occupancy; tapered, they drain over one board time.  Fluid picture: with S resident warps, S/3 of the
// 3-board CTAs finish per board time, so S/3 two-board CTAs and then S/3 one-board CTAs keep every slot busy until
// one board time before the end; board times vary, and twice that share measured best
// (profiles/r02an_taper_sweep.txt, C2 kernel: no taper 109.8 us, 1x 107.7, 1.5x 106.9, 2x 106.7, 3x 107.3 us =
// 6.27 -> 6.45 TB/s; C4, a 1.7 ms launch: 1710 -> 1705 us).
static inline int grid_for(EnvParams &q, int resident_warps_per_sm)
{
    const long long n = q.n;
    const long long S = (long long)sm_count() * resident_warps_per_sm;
    long long n2 = 0, n1 = 0;                           // boards handled by 2-board and by 1-board warps
    if (n >= 8 * S) {                                   // from eight waves on (measured at 18 and 148 waves)
        n1 = S / ENV_BPW * 2;
        n2 = 2 * n1;
    }
    q.seg_na = n - n2 - n1;
    q.seg_wa = (q.seg_na + ENV_BPW - 1) / ENV_BPW;
    q.seg_nb = q.seg_na + n2;
    q.seg_wb = (n2 + 1) / 2;
    long long blocks = q.seg_wa + q.seg_wb + n1;       // one warp per CTA
    if (blocks < 1) blocks = 1;
    if (blocks > 0x7fffffffLL) blocks = 0x7fffffffLL;
    return (int)blocks;
}

// Step launches use the next-board-prefetch instantiation (80 registers); reset / encode the plain one.
// (Prefetch at 64 registers, no prefetch at 64 and at 48 registers were measured slower and dropped.)
template <int MODE, int CW, int CHW>
static void launch_shape(const EnvParams &p, int grid, cudaStream_t s)
{
    if (MODE != MODE_STEP)
        env_kernel<MODE, CW, CHW, false, 4><<<grid, 32, 0, s>>>(p);
    else
        env_kernel<MODE, CW, CHW, true, 3><<<grid, 32, 0, s>>>(p);
}

template <int MODE>
static int launch_env(const EnvParams &p_in, cudaStream_t s)
{
    if (p_in.n == 0) return MSW_OK;
    EnvParams p = p_in;
    const int grid = grid_for(p, MODE == MODE_STEP ? 24 : 32);     // 80 / 64 registers: 24 / 32 one-warp CTAs per SM
    if (p.W == 16 && p.HW == 256)
        launch_shape<MODE, 16, 256>(p, grid, s);       // BASELINE configs 1-3, 5
    else if (p.W == 30 && p.HW == 480)
        launch_shape<MODE, 30, 480>(p, grid, s);       // BASELINE config 4 (Expert, H=16 W=30)
    else if (p.W == 16 && p.HW == 480)
        launch_shape<MODE, 16, 480>(p, grid, s);       // Expert transposed (H=30 W=16)
    else
        launch_shape<MODE, 0, 0>(p, grid, s);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

}  // namespace msw

using namespace msw;

extern "C" int msw_reset(const msw_env_desc *desc, const msw_state *st, int64_t n,
                         const msw_encode_out *out, void *stream)
{
    EnvParams p;
    int rc = fill_params(p, desc, st, n);
    if (rc) return rc;
    if ((rc = set_encode_out(p, out, false))) return rc;
    return launch_env<MODE_RESET>(p, (cudaStream_t)stream);
}

extern "C" int msw_encode(const msw_env_desc *desc, const msw_state *st, int64_t n,
                          const msw_encode_out *out, void *stream)
{
    EnvParams p;
    int rc = fill_params(p, desc, st, n);
    if (rc) return rc;
    if ((rc = set_encode_out(p, out, true))) return rc;
    return launch_env<MODE_ENCODE>(p, (cudaStream_t)stream);
}

static int fill_step(EnvParams &p, const msw_env_desc *desc, const msw_state *st, const msw_step_io *io, int64_t n)
{
    int rc = fill_params(p, desc, st, n);
    if (rc) return rc;
    if (!io) return fail(MSW_ERR_NULL, "io is NULL");
    if (io->rand_mode < 0 || io->rand_mode > 2) return fail(MSW_ERR_ARG, "rand_mode must be 0, 1 or 2");
    if (!io->rand_mode && (io->actions32 != nullptr) == (io->actions64 != nullptr))
        return fail(MSW_ERR_ARG, "exactly one of actions32/actions64 must be set");
    if (!io->reward || !io->done) return fail(MSW_ERR_NULL, "reward/done outputs are required");
    if ((io->inject_sel != nullptr) != (io->inject_bits != nullptr))
        return fail(MSW_ERR_ARG, "inject_bits and inject_sel must be given together");
    p.a32 = io->actions32;
    p.a64 = reinterpret_cast<const long long *>(io->actions64);
    p.rand_mode = io->rand_mode; p.rand_step = io->rand_step;
    p.rk0 = (uint32_t)io->rand_seed; p.rk1 = (uint32_t)(io->rand_seed >> 32);
    p.a_out = io->actions_out32;
    p.inj_bits = io->inject_bits; p.inj_sel = io->inject_sel;
    p.reward = io->reward; p.done = io->done; p.outcome = io->outcome;
    p.new_reveals = io->new_reveals; p.step = io->step; p.rcount = io->revealed_count;
    return set_encode_out(p, &io->enc, false);
}

extern "C" int msw_step(const msw_env_desc *desc, const msw_state *st, const msw_step_io *io,
                        int64_t n, void *stream)
{
    EnvParams p;
    int rc = fill_step(p, desc, st, io, n);
    if (rc) return rc;
    return launch_env<MODE_STEP>(p, (cudaStream_t)stream);
}

extern "C" int msw_step_host(const msw_env_desc *desc, const msw_state *st, const msw_step_io *io,
                             const int32_t *h_actions32, const msw_host_out *h, int64_t n, void *stream)
{
    EnvParams p;
    int rc = fill_step(p, desc, st, io, n);
    if (rc) return rc;
    if (!h_actions32 || !io->actions32) return fail(MSW_ERR_NULL, "msw_step_host needs h_actions32 and io->actions32 staging");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)n, HW = (size_t)p.HW;

    struct Copy { void *dst; const void *src; size_t bytes; };
    Copy copies[8] = {};
    int nc = 0;
    // Queue a device->host copy; a copy that continues the previous one on both sides is merged into it
    // (the Python mirror lays reward|done|... out back to back, so the scalars travel as one DMA).
    auto d2h = [&](void *dst, const void *src, size_t bytes) {
        if (nc && (const char *)copies[nc - 1].src + copies[nc - 1].bytes == (const char *)src &&
            (char *)copies[nc - 1].dst + copies[nc - 1].bytes == (char *)dst)
            copies[nc - 1].bytes += bytes;
        else
            copies[nc++] = {dst, src, bytes};
    };
#define MSW_HOST_SCALAR(field, dev, type, bytes)                                                           \
    if (h && h->field) {                                                                                   \
        if (!(dev)) return fail(MSW_ERR_NULL, "host output " #field " requested without device staging"); \
        d2h(h->field, dev, bytes);                                                                         \
    }
    const bool expand = h && (h->obs || h->mask);
    const size_t wpb = (size_t)p.wpb;
    if (expand) {
        if (!h->stage) return fail(MSW_ERR_NULL, "msw_step_host: host obs/mask requested without the pinned state staging area");
        if (h->shadow && !(h->obs && h->mask))
            return fail(MSW_ERR_NULL, "msw_step_host: a shadow describes BOTH result arrays: obs and mask are required with it");
    }
    MSW_HOST_SCALAR(reward, p.reward, float, N * 4)
    MSW_HOST_SCALAR(done, p.done, uint8_t, N)
    MSW_HOST_SCALAR(outcome, p.outcome, int8_t, N)
    MSW_HOST_SCALAR(new_reveals, p.new_reveals, int32_t, N * 4)
    MSW_HOST_SCALAR(step, p.step, int32_t, N * 4)
    MSW_HOST_SCALAR(revealed_count, p.rcount, int32_t, N * 4)
#undef MSW_HOST_SCALAR

    // (Letting the kernel read the actions from / write the scalars to mapped pinned memory was measured and lost:
    // 196 / 213 / 276 us per step against 155 us with two DMAs, profiles/r01e_e2e_transfer_plans.txt -- removed.)
    MSW_CUDA_TRY(cudaMemcpyAsync(const_cast<int32_t *>(io->actions32), h_actions32, N * 4, cudaMemcpyHostToDevice, s));
    if ((rc = launch_env<MODE_STEP>(p, s))) return rc;
    for (int i = 0; i < nc; ++i)
        MSW_CUDA_TRY(cudaMemcpyAsync(copies[i].dst, copies[i].src, copies[i].bytes, cudaMemcpyDeviceToHost, s));
    if (!expand) {
        MSW_CUDA_TRY(cudaStreamSynchronize(s));
        return MSW_OK;
    }
    // Reference-shaped observation / mask on the host: NOT copied (41*HW bytes per env would make the call
    // PCIe-bound); the packed post-step state they are a pure function of -- the mine and revealed bitboards,
    // 2*wpb words per env; first_click_done is implied (a cell can only be revealed after the first click,
    // env.py:119-122, so revealed != 0 <=> first_click_done wherever it matters) -- is copied into the caller's
    // pinned staging area and expanded on the host (msw_host_expand.cpp).  The copy travels in up to four slices
    // with an event after each, so the host expands slice k while slices k+1.. are still on the bus.
    uint32_t *h_mines = reinterpret_cast<uint32_t *>(h->stage), *h_rev = h_mines + N * wpb;
    constexpr int MAX_SLICES = 4;
    const int slices = N >= 32768 ? MAX_SLICES : 1;
    const size_t per = ((N + slices - 1) / slices + 127) / 128 * 128;
    cudaEvent_t ev[MAX_SLICES] = {};
    int made = 0;
    cudaError_t err = cudaSuccess;
    for (int k = 0; k < slices && err == cudaSuccess; ++k) {
        const size_t lo = (size_t)k * per, hi = lo + per < N ? lo + per : N;
        if (lo >= hi) break;
        err = cudaMemcpyAsync(h_mines + lo * wpb, st->mines + lo * wpb, (hi - lo) * wpb * 4, cudaMemcpyDeviceToHost, s);
        if (err == cudaSuccess)
            err = cudaMemcpyAsync(h_rev + lo * wpb, st->revealed + lo * wpb, (hi - lo) * wpb * 4, cudaMemcpyDeviceToHost, s);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&ev[k], cudaEventDisableTiming);
        if (err == cudaSuccess) {
            ++made;
            err = cudaEventRecord(ev[k], s);
        }
    }
    for (int k = 0; k < made && err == cudaSuccess; ++k) {
        const size_t lo = (size_t)k * per, hi = lo + per < N ? lo + per : N;
        err = cudaEventSynchronize(ev[k]);
        if (err == cudaSuccess)
            expand_obs_host(p.H, p.W, h_mines + lo * wpb, h_rev + lo * wpb, nullptr, (long long)(hi - lo),
                            h->obs ? h->obs + lo * MSW_OBS_CHANNELS * HW : nullptr, h->mask ? h->mask + lo * HW : nullptr,
                            h->shadow ? h->shadow + lo * (size_t)msw_shadow_words(p.H, p.W) : nullptr, h->shadow_valid, h->threads);
    }
    for (int k = 0; k < made; ++k) cudaEventDestroy(ev[k]);
    if (err != cudaSuccess) {
        cudaStreamSynchronize(s);                    // nothing of this call may still be in flight when it returns
        return cuda_fail(err, "msw_step_host: state copy / expansion");
    }
    MSW_CUDA_TRY(cudaStreamSynchronize(s));
    return MSW_OK;
}

extern "C" int msw_unpack_state(const msw_env_desc *desc, const msw_state *st, int64_t n, uint8_t *mine,
                                uint8_t *revealed, uint8_t *flags, uint8_t *counts, void *stream)
{
    UnpackParams q;
    int rc = fill_params(q.e, desc, st, n);
    if (rc) return rc;
    q.o_mine = mine; q.o_rev = revealed; q.o_flags = flags; q.o_counts = counts;
    if (n == 0) return MSW_OK;
    unpack_kernel<<<(unsigned)((n + 7) / 8), 256, 0, (cudaStream_t)stream>>>(q);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

extern "C" int msw_random_actions(const msw_env_desc *desc, const msw_state *st, int64_t n, uint64_t seed,
                                  uint32_t step_index, int32_t valid_only, int32_t *a32, int64_t *a64,
                                  void *stream)
{
    EnvParams e;
    int rc = fill_params(e, desc, st, n);
    if (rc) return rc;
    if (!a32 && !a64) return fail(MSW_ERR_NULL, "no action output given");
    if (n == 0) return MSW_OK;
    ActParams p;
    p.revealed = st->revealed; p.HW = e.HW; p.wpb = e.wpb; p.n = n; p.env_id_base = desc->env_id_base;
    p.k0 = (uint32_t)seed; p.k1 = (uint32_t)(seed >> 32); p.step_index = step_index;
    p.valid_only = valid_only; p.a32 = a32; p.a64 = reinterpret_cast<long long *>(a64);
    random_actions_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

extern "C" int msw_late_start(const msw_env_desc *desc, const msw_state *st, int64_t n, const uint8_t *sel,
                              uint64_t late_seed, float prob, int32_t min_hidden, int32_t max_hidden,
                              int32_t max_attempts, int32_t max_extra_steps, void *stream)
{
    LateParams q;
    int rc = fill_params(q.e, desc, st, n);
    if (rc) return rc;
    if (!(prob >= 0.0f) || min_hidden < 1 || max_hidden < min_hidden || max_attempts < 1 || max_extra_steps < 1)
        return fail(MSW_ERR_ARG, "msw_late_start: bad parameters (prob=%f hidden=[%d,%d] attempts=%d extra=%d)",
                    prob, min_hidden, max_hidden, max_attempts, max_extra_steps);
    if (n == 0 || prob <= 0.0f) return MSW_OK;
    q.sel = sel;
    q.lk0 = (uint32_t)late_seed; q.lk1 = (uint32_t)(late_seed >> 32);
    const double p24 = (double)prob * 16777216.0;
    q.prob24 = p24 >= 16777216.0 ? 16777216u : (uint32_t)p24;
    q.min_hidden = min_hidden; q.max_hidden = max_hidden;
    q.max_attempts = max_attempts; q.max_extra_steps = max_extra_steps;
    late_start_kernel<<<(unsigned)((n + 3) / 4), 128, 0, (cudaStream_t)stream>>>(q);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

extern "C" int msw_gather_encode(const msw_env_desc *desc, const uint32_t *snap_mines, const uint32_t *snap_revealed,
                                 const uint32_t *snap_flags, const uint8_t *snap_first, int64_t rows_in,
                                 const int64_t *idx, int64_t m, const msw_encode_out *out, void *stream)
{
    if (!snap_mines || !snap_revealed || !snap_first || !idx) return fail(MSW_ERR_NULL, "msw_gather_encode: NULL pointer");
    if (rows_in < 1) return fail(MSW_ERR_BAD_SHAPE, "msw_gather_encode: rows_in=%lld", (long long)rows_in);
    GatherParams q;
    int rc = fill_geometry(q.e, desc, m);
    if (rc) return rc;
    if ((rc = set_encode_out(q.e, out, true))) return rc;
    q.e.flags = const_cast<uint32_t *>(snap_flags);           // encoder consults flags only when present
    q.s_mines = snap_mines; q.s_revealed = snap_revealed; q.s_flags = snap_flags; q.s_first = snap_first;
    q.idx = reinterpret_cast<const long long *>(idx); q.rows_in = rows_in;
    if (m == 0) return MSW_OK;
    long long blocks = (m + 7) / 8;
    const long long cap = (long long)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    cudaStream_t st = (cudaStream_t)stream;
    if (q.e.W == 16 && q.e.HW == 256)
        gather_encode_kernel<16, 256><<<(unsigned)blocks, 256, 0, st>>>(q);
    else
        gather_encode_kernel<0, 0><<<(unsigned)blocks, 256, 0, st>>>(q);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}

extern "C" int msw_forced_subset(const msw_env_desc *desc, const msw_state *st, int64_t n, uint32_t *out_bits,
                                 void *stream)
{
    SubsetParams q;
    int rc = fill_params(q.e, desc, st, n);
    if (rc) return rc;
    if (!out_bits) return fail(MSW_ERR_NULL, "msw_forced_subset: out_bits is NULL");
    q.out = out_bits;
    if (n == 0) return MSW_OK;
    const size_t smem = 4 * (3 * (size_t)MSW_MAX_CELLS + 128);
    subset_reveal_kernel<<<(unsigned)((n + 3) / 4), 128, smem, (cudaStream_t)stream>>>(q);
    MSW_CUDA_TRY(cudaGetLastError());
    return MSW_OK;
}
