/*
 * msw_b200.h -- C ABI of the B200-native minesweeper-ppo rollout hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI
 * layer -- its boundary is the duck-typed Python API of minesweeper/env.py and
 * minesweeper/buffers.py -- so each entry point below names the reference
 * function it replaces; minesweeper_ppo_b200/{env,buffers}.py bind them with
 * ctypes behind the reference's own class and method names (INTEGRATION.md).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch types.
 *   - "device" pointers are CUDA device memory owned by the caller (PyTorch's
 *     caching allocator); the library never allocates or frees device memory
 *     and keeps no global state except a thread-local last-error string.
 *   - Every device entry point is an asynchronous, stream-ordered launch on
 *     `stream` (a cudaStream_t passed as void*); no host synchronisation
 *     inside.  The *_host entry points take pinned HOST buffers, copy in/out on
 *     `stream` and synchronise it before returning.
 *   - Return value: 0 on success, MSW_ERR_* (>0) on bad arguments, or a
 *     negated cudaError_t (<0) when the CUDA runtime reports an error;
 *     msw_last_error() describes the most recent failure on this thread.
 *   - There is no CPU fallback anywhere behind this interface.
 *
 * Board layout: a board is a flat bitstring of H*W cells, cell (r,c) at bit
 * r*W+c, stored as msw_words_per_board(H,W) little-endian uint32 words
 * (== np.packbits(board.reshape(-1), bitorder="little") padded to 4 bytes).
 * Limits: 1 <= W <= 32, 1 <= H*W <= 1024, 0 <= mine_count <= H*W-1.
 */
#ifndef MSW_B200_H
#define MSW_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSW_VERSION 1
#define MSW_OBS_CHANNELS 10        /* env.py:79-85: revealed + one-hot counts 0..8 */
#define MSW_MAX_CELLS 1024

enum {
    MSW_OK = 0,
    MSW_ERR_BAD_SHAPE = 1,         /* H, W, mine_count or n out of range */
    MSW_ERR_NULL = 2,              /* required pointer is NULL */
    MSW_ERR_ALIGN = 3,             /* pointer not aligned for vector stores */
    MSW_ERR_ARG = 4                /* inconsistent arguments */
};

/* Static description of one shard of environments; mirrors EnvConfig
 * (minesweeper/env.py:19-30) plus what VecMinesweeper.__init__ (env.py:382-403)
 * derives from `seed`. */
typedef struct msw_env_desc {
    int32_t H, W;
    int32_t mine_count;
    int32_t safe_nbhd;             /* EnvConfig.guarantee_safe_neighborhood */
    /* Rewards pre-rounded to fp32 exactly as the reference does: accumulated in
     * float64 (env.py:110,128,137,142) then stored into a float32 array
     * (env.py:483,501).  step = -step_penalty; loss = loss_reward-step_penalty;
     * win = win_reward-step_penalty. */
    float reward_step, reward_loss, reward_win;
    int32_t reserved;
    uint64_t seed;                 /* key of the counter-based board sampler */
    int64_t env_id_base;           /* global id of env 0 (multi-GPU sharding) */
} msw_env_desc;

/* Persistent per-env state (device).  Replaces the MinesweeperEnv attributes
 * mine_mask / revealed / flags / first_click_done / step_count /
 * _last_new_reveals (env.py:68-75); adjacent_counts is recomputed from
 * `mines` on the fly and never stored. */
typedef struct msw_state {
    uint32_t *mines;               /* [n][wpb] */
    uint32_t *revealed;            /* [n][wpb] */
    uint32_t *flags;               /* [n][wpb]; NULL == no flags anywhere (hot path) */
    int32_t  *meta;                /* [n][4]: first_click_done, step_count,
                                      episode_idx (sampler counter), last_new_reveals;
                                      16-byte aligned */
} msw_state;

/* Outputs of reset / step / encode (device).  obs must be 16-byte aligned when
 * H*W % 4 == 0 (vector store path); nullable members may be NULL. */
typedef struct msw_encode_out {
    float   *obs;                  /* [n][10][H][W] f32          env.py:172-192 */
    uint8_t *mask;                 /* [n][H*W] bool              env.py:194-196 */
    float   *mine_labels;          /* nullable [n][H][W] f32     train_rl.py:205-212 */
    uint8_t *mine_valid;           /* nullable [n][H][W] bool    train_rl.py:205-212 */
} msw_encode_out;

typedef struct msw_step_io {
    const int32_t *actions32;      /* [n]; exactly one of actions32/actions64 */
    const int64_t *actions64;      /* [n] */
    const uint32_t *inject_bits;   /* nullable [n][wpb]: layouts for parity tests */
    const uint8_t  *inject_sel;    /* nullable [n]: 1 => env takes inject_bits when it
                                      places mines in this step */
    float   *reward;               /* [n] f32   env.py:501 */
    uint8_t *done;                 /* [n] bool  env.py:502 */
    int8_t  *outcome;              /* nullable [n]: 0 none, 1 win, 2 loss  env.py:493 */
    int32_t *new_reveals;          /* nullable [n]: aux.last_new_reveals (pre-reset) */
    int32_t *step;                 /* nullable [n]: aux.step (pre-reset) */
    int32_t *revealed_count;       /* nullable [n]: popcount(revealed) (pre-reset);
                                      revealed_frac = count / (H*W), env.py:165 */
    msw_encode_out enc;            /* observation of the post-(auto-)reset state */
    /* Built-in synthetic policy for env-only throughput runs (BASELINE.md section 4): when
     * rand_mode != 0 the actions are NOT read from actions32/64 (both may be NULL) but drawn
     * inside the step launch exactly as msw_random_actions(seed=rand_seed, step_index=rand_step,
     * valid_only = rand_mode == 1) would draw them, and written to actions_out32 (nullable). */
    int32_t  rand_mode;            /* 0 off, 1 uniformly random unrevealed cell, 2 any cell */
    uint32_t rand_step;
    uint64_t rand_seed;
    int32_t *actions_out32;        /* nullable [n] */
} msw_step_io;

int msw_version(void);
const char *msw_last_error(void);
int msw_words_per_board(int32_t H, int32_t W);

/* VecMinesweeper.reset (env.py:468-477) -> MinesweeperEnv.reset (env.py:87-101):
 * zero all state, bump the sampler counter, emit the all-zero observation and
 * all-true mask.  No mines are placed at reset. */
int msw_reset(const msw_env_desc *desc, const msw_state *st, int64_t n,
              const msw_encode_out *out, void *stream);

/* VecMinesweeper.step (env.py:479-511) with everything under it fused into one
 * launch: MinesweeperEnv.step (env.py:103-152), _place_mines_safe (:280-312),
 * _compute_adjacent_counts (:314-335), flood_fill_reveal (env_numba.py:16-77),
 * auto-reset (:497-498), _build_obs (:172-192), _compute_action_mask (:194-196),
 * _build_aux (:163-170) and the aux label extraction of train_rl.py:203-219. */
int msw_step(const msw_env_desc *desc, const msw_state *st, const msw_step_io *io,
             int64_t n, void *stream);

/* _build_obs / _compute_action_mask of the current state without stepping. */
int msw_encode(const msw_env_desc *desc, const msw_state *st, int64_t n,
               const msw_encode_out *out, void *stream);

/* Expands the bitboards into the reference's per-cell arrays for the
 * `vec.envs[i]` compatibility views (env.py:68-71): bool [n][H*W] each and
 * adjacent_counts u8 [n][H*W] (env.py:314-335).  Any output may be NULL. */
int msw_unpack_state(const msw_env_desc *desc, const msw_state *st, int64_t n,
                     uint8_t *mine, uint8_t *revealed, uint8_t *flags,
                     uint8_t *counts, void *stream);

/* VecMinesweeper._apply_late_start (env.py:416-466; SURVEY section 8 row f3) for
 * freshly reset boards (all of them, or those with sel[i] != 0 -- pass the
 * `done` output of msw_step): with probability `prob` pre-play random safe
 * cells until at most target_hidden in [min_hidden, max_hidden] safe cells stay
 * hidden, retrying up to max_attempts times and leaving the board fresh on
 * failure.  Randomness: counter-based Philox stream keyed by late_seed (the
 * reference's shared sequential NumPy generator is not reproducible in
 * parallel).  Call msw_encode afterwards to observe the resulting boards. */
int msw_late_start(const msw_env_desc *desc, const msw_state *st, int64_t n,
                   const uint8_t *sel, uint64_t late_seed, float prob,
                   int32_t min_hidden, int32_t max_hidden, int32_t max_attempts,
                   int32_t max_extra_steps, void *stream);

/* Compact replay + fused minibatch gather (SURVEY section 8 row f2), replacing the
 * obs / action_mask / mine_labels / mine_valid index gathers of
 * RolloutBuffer.get_minibatches (buffers.py:96-116): transitions are stored as
 * bitboard snapshots (snap_mines / snap_revealed / nullable snap_flags
 * [rows_in][wpb], snap_first [rows_in]) and row j of the minibatch is re-encoded
 * from snapshot idx[j] straight into `out` (m rows).  Bit-identical to gathering
 * rows of a dense buffer. */
int msw_gather_encode(const msw_env_desc *desc, const uint32_t *snap_mines,
                      const uint32_t *snap_revealed, const uint32_t *snap_flags,
                      const uint8_t *snap_first, int64_t rows_in, const int64_t *idx,
                      int64_t m, const msw_encode_out *out, void *stream);

/* rules.analyze_forced_modules (rules.py:206-259; SURVEY section 8 row f4): the
 * pairwise subset rule on ground-truth mines, for every env at once.  out_bits
 * [n][wpb] receives the bitboard of "subset_reveal" cells (cells proven safe
 * because two number cells with nested unknown-neighbour sets hold the same
 * number of mines). */
int msw_forced_subset(const msw_env_desc *desc, const msw_state *st, int64_t n,
                      uint32_t *out_bits, void *stream);

/* avoidability.analyze_avoidability (avoidability.py:145-394; SURVEY section 8
 * row f4) for every env at once: frontier components, unit + subset rules and,
 * when those find no safe cell, the exact per-component feasibility search.
 * safe_bits [n][wpb]: bitboard of forced_safe_cells; comp_of_cell [n][H*W]:
 * smallest cell index of the frontier component a cell belongs to (-1 off the
 * frontier); comp_size [n][H*W]: size of the component whose smallest cell is
 * that index (0 elsewhere) -- the non-zero entries in index order are the
 * reference's component_sizes list; flags [n]: bit 0 avoidable, bit 1 frontier
 * non-empty, bit 2 first_click_done, bit 3 the exact search ran out of its
 * per-lane step budget (search_budget, 0 = default 2^23; the cells it could
 * not decide are reported as not safe).  The chosen-cell fields of the
 * reference's result follow from these arrays: chosen_is_forced_safe =
 * safe[chosen], chosen_component_size = comp_size[comp_of_cell[chosen]]. */
int msw_avoidability(const msw_env_desc *desc, const msw_state *st, int64_t n,
                     uint32_t *safe_bits, int16_t *comp_of_cell, int16_t *comp_size,
                     uint8_t *flags, uint32_t search_budget, void *stream);

/* Synthetic action source for benchmarks/tests (BASELINE.md section 4): a
 * uniformly random unrevealed cell per env (valid_only=1; 0 if none) or a
 * uniformly random cell (valid_only=0).  Writes whichever of a32/a64 is
 * non-NULL. */
int msw_random_actions(const msw_env_desc *desc, const msw_state *st, int64_t n,
                       uint64_t seed, uint32_t step_index, int32_t valid_only,
                       int32_t *a32, int64_t *a64, void *stream);

/* RolloutBuffer.compute_gae (buffers.py:78-94) over time-major [T][N] fp32
 * with unfused IEEE multiplies/adds in the reference's order.  gamma_f32 and
 * gamma_lam_f32 are float(gamma) and float(gamma*lam) (product in float64).
 * last_values_prescaled != 0: `last_values` already holds gamma*last_value as
 * the caller's tensor dtype rounds it (the reference's bootstrap value is fp16
 * under CUDA autocast, train_rl.py:272-277, so `gamma * next_value` at t=T-1 is
 * rounded to fp16 before it is promoted, buffers.py:88-90); the kernel then
 * skips that one multiply. */
int msw_gae(const float *rewards, const float *values, const uint8_t *dones,
            const float *last_values, float *advantages, float *returns,
            int64_t T, int64_t N, float gamma_f32, float gamma_lam_f32,
            int32_t last_values_prescaled, void *stream);

/* Fused masked categorical sampler (SURVEY section 8 row f1), replacing
 * train_rl.py:229-235 + the int64->int32 conversion of :239: logits [n][A]
 * (logits_dtype 0 = f32, 1 = f16, 2 = bf16) are masked with the reference's
 * fill value (-1e9 for f32, -1e4 for half types), soft-maxed in fp32, one
 * action per row is drawn by inverse CDF with a Philox uniform keyed by
 * (seed, row_id_base + row, step_index), and log_prob(action) is returned.
 * `epoch` (nullable device uint32) is added to the high word of step_index when
 * the kernel runs, so a captured CUDA graph draws fresh numbers on each replay.
 * Writes whichever of actions64 / actions32 / logp is non-NULL.  `mask` is in/out
 * for one case only: a row without any legal action is made all-legal (and
 * sampled as such), the collector's guard of train_rl.py:166-168 / 263-265. */
int msw_masked_sample(const void *logits, int32_t logits_dtype, uint8_t *mask,
                      int64_t n, int32_t A, uint64_t seed, uint64_t step_index,
                      const uint32_t *epoch, int64_t row_id_base, int64_t *actions64,
                      int32_t *actions32, float *logp, void *stream);

/* Greedy action of the evaluator (eval.py:330-340): actions[r] = the argmax of
 * logits.masked_fill(~mask, -1e9) over row r of fp32 logits [n][A], exactly as
 * torch's argmax picks it -- masked cells compete at -1e9, ties go to the first
 * index, a NaN wins (the first NaN).  `mask` (bool [n][A]) is in/out for one
 * case only: a row without any legal action is made all-legal first (the guard
 * of eval.py:336-338).  One warp per row. */
int msw_masked_argmax(const float *logits, uint8_t *mask, int64_t n, int32_t A,
                      int32_t *actions, void *stream);

/* Episode accounting of eval.evaluate_vec (eval.py:350-428) on the device, as
 * two launches around msw_step.  `counters` is int64 [MSW_EVAL_COUNTERS]
 * (zero, except MSW_EVAL_ERROR_KEY = INT64_MAX, at the start of an evaluation);
 * updates are integer atomics, so the totals do not depend on the order. */
enum {
    /* msw_eval_pre_step */
    MSW_EVAL_INVALID = 0,              /* picks outside the mask, over all n envs */
    MSW_EVAL_FORCED_STEPS, MSW_EVAL_FORCED_CORRECT,      /* chosen cell in subset_reveal */
    MSW_EVAL_GUESS_ATTEMPTS, MSW_EVAL_GUESS_SUCCESS,     /* chosen cell not in it */
    MSW_EVAL_REVEAL_TOTAL,             /* analysed envs with first_click_done */
    MSW_EVAL_FORCED_GUESS_TOTAL, MSW_EVAL_FORCED_GUESS_SUCCESS,
    MSW_EVAL_SAFE_OPTION_TOTAL, MSW_EVAL_SAFE_OPTION_HITS, MSW_EVAL_SAFE_OPTION_MISSES,
    MSW_EVAL_SAFE_CELLS,               /* sum of count_forced_safe_cells */
    MSW_EVAL_COMP_SIZE_SUM, MSW_EVAL_COMP_COUNT,         /* component_sizes */
    MSW_EVAL_CHOSEN_SIZE_SUM, MSW_EVAL_CHOSEN_COUNT,     /* chosen_component_size */
    MSW_EVAL_PRE_COUNTERS,
    /* msw_eval_post_step */
    MSW_EVAL_WINS = MSW_EVAL_PRE_COUNTERS, MSW_EVAL_TOTAL_STEPS,
    MSW_EVAL_NEW_REVEALS,              /* sum of last_new_reveals of uncounted envs */
    MSW_EVAL_FORCED_GUESS_EPISODES,
    /* smallest step_index * n + env of an analysed env whose msw_avoidability
     * flag bit 3 (search budget exceeded) was set; INT64_MAX if none */
    MSW_EVAL_ERROR_KEY,
    MSW_EVAL_COUNTERS
};

/* Before msw_step, on the state the actions were chosen on: for every env, an
 * invalid pick (mask[i][actions[i]] == 0) is counted; envs with counted[i] == 0
 * and i < batch_size are analysed -- the `safe` test on the mines, subset-rule
 * hit or guess from msw_forced_subset's subset_bits, and, when
 * first_click_done, the avoidability bookkeeping of avoidability.py:41-49 from
 * msw_avoidability's arrays (safe_bits, comp_of_cell, comp_size, avoid_flags),
 * which sets ep_unavoidable[i] for a forced guess.  belief_sel (nullable, u8
 * [n][H*W]) is rewritten whole: 1 + mine for each unknown (not revealed, not
 * flagged) cell of an analysed env, 0 elsewhere. */
int msw_eval_pre_step(const msw_env_desc *desc, const msw_state *st, int64_t n, int64_t batch_size,
                      const int32_t *actions, const uint8_t *mask, const uint32_t *subset_bits,
                      const uint32_t *safe_bits, const int16_t *comp_of_cell, const int16_t *comp_size,
                      const uint8_t *avoid_flags, const uint8_t *counted, uint8_t *ep_unavoidable,
                      uint8_t *belief_sel, int64_t *counters, int64_t step_index, void *stream);

/* After msw_step, over all n envs (eval.py:405-428): step_counter[i] += 1; an
 * uncounted env adds its last_new_reveals; an uncounted env that is done (or,
 * when max_steps > 0, has reached max_steps) adds its steps (and, if done, its
 * win and ep_unavoidable), resets its step counter, becomes counted and adds 1
 * to *finished. */
int msw_eval_post_step(int64_t n, const uint8_t *done, const int8_t *outcome, const int32_t *new_reveals,
                       uint8_t *counted, int32_t *step_counter, const uint8_t *ep_unavoidable,
                       int32_t max_steps, int64_t *counters, int32_t *finished, void *stream);

/* Fused GroupNorm + (fp32 residual add) + ReLU + Dropout2d between the cuDNN
 * convolutions of the rollout forward (SURVEY section 8 row f4; replaces the
 * eager norm/act/dropout/add/cast kernels of cnn_residual.py:17-27, 50-54
 * under the fp16 autocast of train_rl.py:222).  x16: fp16 NHWC [n][HW][C] conv
 * output WITHOUT its bias; conv_bias (nullable, fp32 [C]) is added before the
 * norm; statistics and arithmetic in fp32; y16 (fp16 NHWC, the next conv's
 * input) and/or y32 (fp32 NHWC, the residual stream) are written.  Needs
 * C % 8 == 0 and (C/G) % 8 == 0; drop_p > 0 applies a Dropout2d channel mask
 * keyed by (seed, call_id [+ *epoch in the high word], sample_id_base + sample,
 * channel) -- the GLOBAL sample index, so masks do not depend on how envs are
 * sharded over GPUs -- and is only allowed without res32.  pool32 (nullable, fp32 [n][C]) receives the
 * mean over HW of the fp32 output -- the AdaptiveAvgPool2d(1) that opens the
 * value head (cnn_residual.py:65) -- so the last block need not write y32. */
int msw_gn_act(const void *x16, const float *conv_bias, const float *res32,
               const float *gamma, const float *beta,
               void *y16, float *y32, int64_t n, int32_t HW, int32_t C, int32_t G,
               float eps, int32_t relu, float drop_p, uint64_t seed, uint64_t call_id,
               const uint32_t *epoch, float *save_mean, float *save_rstd,
               uint8_t *save_mask, float *pool32, int64_t sample_id_base, void *stream);

/* Input of the stem convolution: fp32 NCHW observation planes obs [n][Cin][HW] (Cin <= 16; the env's 10
 * planes) -> fp16 NHWC out16 [n][HW][16] with the missing channels zero, i.e. the autocast cast of
 * train_rl.py:222 and the channel padding the tensor-core convolution needs, in one pass. */
int msw_pack_obs16(const float *obs, void *out16, int64_t n, int32_t Cin, int32_t HW, void *stream);

/* Both per-cell heads of CNNResidualPolicy (cnn_residual.py:57-62, 73-77,
 * 87-94: 1x1 conv C->C, ReLU, 1x1 conv C->1, for the policy and for the mine
 * belief) in one launch over the fp16 NHWC trunk activation a16 [rows][C],
 * rows = n*H*W.  w1 [2C][C] / b1 [2C]: first-layer weights and biases, policy
 * units first; w2 [2C] / b2 [2]: second-layer weights and biases; all fp16, as
 * the fp16 autocast of train_rl.py:222 casts them.  fp32 accumulation, hidden
 * activations rounded to fp16 before the ReLU as the reference's conv output
 * is.  Writes fp16 out_policy [rows] (= logits [n][H*W]) and out_mine [rows]
 * (= mine logits [n][1][H][W]).  C in {32, 64, 96, 128}. */
int msw_cell_heads(const void *a16, const void *w1, const void *b1, const void *w2,
                   const void *b2, void *out_policy, void *out_mine, int64_t rows,
                   int32_t C, void *stream);

/* 3x3 "same" convolution of the policy trunk (cnn_residual.py:10-13: Conv2d(C, C, 3, padding=1); :50: the
 * stem Conv2d(10, C, 3, padding=1) on the 16-channel input of msw_pack_obs16) on the tcgen05 tensor cores, for
 * the shapes the medium config and the default residual model use: 16x16 boards, C = 96 (Cin = 96 or 16) or
 * C = 128 (Cin = 128 or 16; each board on a 2-CTA cluster).  x16: fp16 NHWC [n][16][16][Cin];
 * w_taps16: fp16 [9][C][Cin], tap = ky*3 + kx of the module's [C][Cin][3][3] weight (zero for padded input
 * channels); y16: fp16 NHWC conv output WITHOUT bias (msw_gn_act adds it), fp32 accumulation. */
int msw_conv3x3(const void *x16, const void *w_taps16, void *y16, int64_t n, int32_t H, int32_t W,
                int32_t Cin, int32_t C, void *stream);

/* msw_conv3x3 with msw_gn_act fused into its epilogue: one launch for "convolution, GroupNorm, (+ fp32
 * residual), ReLU, Dropout2d" of a residual block half (cnn_residual.py:17-27):
 *   y16 = fp16(relu(GN(fp16(conv(x16)) + conv_bias) [+ res32]) [* Dropout2d]),  y32 (nullable) the same in fp32;
 * the conv output is rounded to fp16 before the norm exactly as the autocast reference does; Dropout2d draws
 * msw_gn_act's stream, keyed by sample_id_base + board.  16x16 boards, groups of 16 channels: C = 96 with G = 6
 * or C = 128 with G = 8; Cin = C or 16 (the stem).
 * res32 (nullable; Cin = C only) and y32 are in the kernels' PRIVATE "P8" order -- [n][tile 2][32-channel slice
 * C/32][8-channel chunk 4][pixel-in-tile 128][8] floats -- in which every 256-bit access of a warp is one contiguous
 * KB (the pixel-major NHWC order costs one line per lane); only this function reads or writes that stream.
 * pool4 (nullable, with res32, instead of y32): fp32 [n][Q][C] partial sums of the fp32 output -- Q = 4 row
 * quarters (C = 96) or 8 = 2 tiles x 4 row quarters (C = 128) -- whose sum over Q / 256 is the
 * AdaptiveAvgPool2d(1) of the value head (cnn_residual.py:65).
 * max_ctas: 0 = one persistent CTA per SM; k > 0 caps the grid (C = 128: rounded down to an even count, one
 * 2-CTA cluster per board at a time) so that two launches on different streams can
 * share the GPU (FusedRolloutForward overlaps an HBM-bound residual layer with an MMA-bound one that way). */
int msw_conv3x3_gn(const void *x16, const void *w_taps16, const float *conv_bias, const float *res32,
                   const float *gamma, const float *beta, void *y16, float *y32, float *pool4, int64_t n,
                   int32_t H, int32_t W, int32_t Cin, int32_t C, int32_t G, float eps, float drop_p,
                   uint64_t seed, uint64_t call_id, const uint32_t *epoch, int64_t sample_id_base, int32_t max_ctas,
                   void *stream);

/* The whole rollout forward of the three-convolution baseline policy (policy.CNNPolicy, build_model("cnn"):
 * conv 3x3 -> ReLU -> GroupNorm(4, 32) -> conv 3x3 -> ReLU -> GroupNorm(8, 64) -> conv 3x3 -> ReLU, then the 1x1
 * policy and mine heads and the value head's average pool) on 16x16 boards in one persistent tcgen05 launch, with
 * the roundings of the fp16 autocast forward (train_rl.py:222-227): each convolution accumulates in fp32, adds its
 * bias and rounds once to fp16; GroupNorm runs in fp32 on the fp16 ReLU output and is rounded to fp16 as the next
 * convolution's input.
 * x16: fp16 NHWC [n][16][16][16] (msw_pack_obs16's layout: observation planes, missing channels zero).
 * wK_taps16: fp16 [9][Cout][Cin], tap = ky*3 + kx of the module's weight (conv1's input channels padded to 16 with
 * zeros).  bK, gammaK, betaK: fp32 conv biases and GroupNorm affine.  wp16 / wm16: fp16 [64] weights of the 1x1
 * policy / mine heads, bp16 / bm16 their fp16 biases (one value each).
 * Writes fp16 logits16 [n][256] and mine16 [n][256] (the heads, fp32 sums over the 64 channels) and pooled16
 * [n][64] (the mean over the board of the fp16 feature map, summed in a fixed order).
 * Only H = W = 16, Cin = 16, widths C1 / C2 / C3 = 32 / 64 / 64 and groups G1 / G2 = 4 / 8; anything else is
 * MSW_ERR_BAD_SHAPE.  x16, the taps, the fp32 vectors and wp16 / wm16 must be 16-byte aligned. */
int msw_cnn_forward(const void *x16, const void *w1_taps16, const float *b1, const float *gamma1, const float *beta1,
                    const void *w2_taps16, const float *b2, const float *gamma2, const float *beta2,
                    const void *w3_taps16, const float *b3, const void *wp16, const void *bp16, const void *wm16,
                    const void *bm16, void *logits16, void *mine16, void *pooled16, int64_t n, int32_t H, int32_t W,
                    int32_t Cin, int32_t C1, int32_t G1, int32_t C2, int32_t G2, int32_t C3, float eps1, float eps2,
                    void *stream);

/* Backward of msw_gn_act for the training forward.  save_mean / save_rstd
 * ([n][G]) and save_mask ([n][HW][C/8], bit k = channel 8j+k passed ReLU and
 * Dropout2d) come from the forward call (all three nullable there, given
 * together).  g16 / g32 are the upstream gradients of y16 / y32 (either may be
 * NULL).  Writes dx16 (gradient of the conv output, fp16), dres32 (nullable,
 * gradient of res32) and per-sample partial sums [n][C] of the gamma / beta /
 * conv-bias gradients, which the caller reduces over n (fixed order, no float
 * atomics). */
int msw_gn_act_bwd(const void *x16, const float *conv_bias, const float *gamma,
                   const float *mean, const float *rstd, const uint8_t *mask,
                   const void *g16, const float *g32, void *dx16, float *dres32,
                   float *part_dgamma, float *part_dbeta, float *part_dbias,
                   int64_t n, int32_t HW, int32_t C, int32_t G, float drop_p,
                   void *stream);

/* Host-buffer form of msw_step for callers that keep the reference's NumPy
 * calling convention (VecMinesweeper.step(actions: np.ndarray), env.py:479):
 * `h_actions32` and the non-NULL per-env scalar outputs are pinned host
 * buffers; `io` holds the device staging buffers (same meaning as msw_step;
 * io->actions32 is the device staging buffer for the actions; io->enc may be
 * all NULL).  Copies actions in, runs the step, copies the requested scalars
 * back and synchronises `stream`.
 *
 * obs / mask (the arrays VecMinesweeper.step returns, env.py:507-510: fp32
 * [n][10][H][W] and bool [n][HW]) are ORDINARY host memory and are not copied
 * over PCIe: the packed post-step state they are a pure function of (the mine
 * and revealed bitboards: 2*wpb words per env, 64 B instead of 10.5 KB at
 * 16x16; first_click_done is implied, see msw_expand_obs_host) is copied into
 * `stage` (pinned, at least n*2*wpb int32: mines, then revealed) in up to
 * four slices and expanded on `threads` host threads (0 = every CPU the
 * process may run on), slice k while slices k+1.. are still on the bus.
 * That is a format conversion of the GPU's result; no game logic runs on the
 * host.  With `shadow` set only what changed since the arrays were last
 * filled is rewritten (delta mode, below). */
typedef struct msw_host_out {
    float   *obs;                  /* nullable; ordinary host memory */
    uint8_t *mask;                 /* nullable; ordinary host memory */
    float   *reward;               /* nullable */
    uint8_t *done;                 /* nullable */
    int8_t  *outcome;              /* nullable */
    int32_t *new_reveals;          /* nullable */
    int32_t *step;                 /* nullable */
    int32_t *revealed_count;       /* nullable */
    int32_t *stage;                /* pinned, required when obs or mask is set */
    int32_t  threads;
    int32_t  shadow_valid;         /* 0: obs / mask hold anything -> everything is written and the shadow initialised;
                                    * != 0: obs / mask hold exactly what `shadow` describes -> only what differs is rewritten */
    uint64_t *shadow;              /* nullable; [n][msw_shadow_words(H, W)] ordinary host memory (see below) */
} msw_host_out;

/* The host-side expansion on its own: packed state arrays IN HOST MEMORY (h_mines / h_revealed int32 [n][wpb],
 * h_meta int32 [n][4], layouts of msw_state; h_meta may be NULL: first_click_done only gates the count planes of
 * REVEALED cells, and a cell can only be revealed after the first click) -> _build_obs (env.py:172-192) / _compute_action_mask
 * (env.py:194-196) arrays in host memory.  Pure host function (no CUDA call), used by msw_step_host and by
 * VecMinesweeper.reset() in the NumPy convention. */
int msw_expand_obs_host(const msw_env_desc *desc, const int32_t *h_mines, const int32_t *h_revealed,
                        const int32_t *h_meta, int64_t n, float *h_obs, uint8_t *h_mask, int32_t threads);

/* Delta mode of the expansion.  A caller that keeps the SAME obs / mask arrays across calls (the Python mirror
 * recycles them from a pool, VecMinesweeper._result_arrays) passes a `shadow`: the 10*H*W bit planes those arrays
 * currently hold (bit p*HW + r*W + c of env i's msw_shadow_words(H, W) little-endian 64-bit words = obs[i][p][r][c],
 * plane 0 = ~mask).  Only the groups of eight values whose bits differ from the shadow are rewritten (a step changes
 * ~10 % of an env's cache lines under random play), then the shadow is updated; the arrays end up byte-identical to
 * the full expansion as long as nobody else wrote to them.  obs, mask and shadow are all required. */
int msw_shadow_words(int32_t H, int32_t W);     /* 64-bit words per env; 0 for an unsupported board */
int msw_expand_obs_host_delta(const msw_env_desc *desc, const int32_t *h_mines, const int32_t *h_revealed,
                              const int32_t *h_meta, int64_t n, float *h_obs, uint8_t *h_mask,
                              uint64_t *shadow, int32_t shadow_valid, int32_t threads);

int msw_step_host(const msw_env_desc *desc, const msw_state *st,
                  const msw_step_io *io, const int32_t *h_actions32,
                  const msw_host_out *h_out, int64_t n, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MSW_B200_H */
