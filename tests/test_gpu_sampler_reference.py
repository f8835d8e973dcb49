"""The fused masked sampler (msw_masked_sample) draw by draw against a float64 inverse CDF.

For every row the host recomputes the kernel's uniform: Philox4x32-10 with the sampler's key and counter layout,
then the float32 mapping of the first word.  The float64 reference is torch's semantics for the collector's
`masked_fill` + `Categorical`: the fill value rounded to the logits' dtype, the softmax, and the first cell whose
cumulative mass exceeds u.  The kernel must return that cell, or, when u lies within BOUNDARY_TOL of a cell
boundary (float32 `expf` and summation order), the cell on the other side of it.

The lane-boundary cases pin a defect of the warp-level selection: the float32 Hillis-Steele scan of the lane sums
is not monotone, so a lane holding no mass can end up one ulp above the lanes before it, and a uniform in that gap
picked the empty lane's first cell -- a masked cell, or, when A is not a multiple of 32, an index past the row."""
import math

import numpy as np
import pytest

FILL = {"float32": -1e9, "float16": -1e4, "bfloat16": -1e4}     # train_rl.py:229-232, before rounding to the dtype
BOUNDARY_TOL = 4e-6          # relative to the row's total mass: float32 expf + summation-order error, with margin
NEAR_BOUNDARY_MAX = 1e-2     # rows with u that close to a boundary (up to 2 * tol per boundary: ~0.4 % at A = 1024)
DECIDED_MAX = 1e-3           # rows whose action is not the float64 cell: a shifted CDF would exceed this
LOGP_ATOL, LOGP_RTOL = 2e-5, 1e-6
M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(k0, k1, c0, c1, c2, c3):
    """Philox4x32-10 over arrays of counters (uint64 arithmetic, 32-bit words); returns the four output words."""
    k0, k1 = np.uint64(k0), np.uint64(k1)
    x0, x1, x2, x3 = (np.array(a, dtype=np.uint64) & M32 for a in np.broadcast_arrays(c0, c1, c2, c3))
    for _ in range(10):
        p0, p1 = x0 * np.uint64(0xD2511F53), x2 * np.uint64(0xCD9E8D57)
        x0, x1, x2, x3 = (p1 >> np.uint64(32)) ^ x1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ x3 ^ k1, p0 & M32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return tuple(a.astype(np.uint32) for a in (x0, x1, x2, x3))


def sampler_w0(seed: int, row_ids, step_index: int, epoch: int = 0) -> np.ndarray:
    """First Philox word of the draw for global rows `row_ids`: key (seed_lo, seed_hi ^ 'SAMP'), counter
    (row_lo, row_hi, step_lo, step_hi + epoch).  The epoch adds to the high word of the step, mod 2^32."""
    rid = np.asarray(row_ids, dtype=np.uint64)
    step = (int(step_index) + (int(epoch) << 32)) & 0xFFFFFFFFFFFFFFFF
    return philox4x32_10(seed & 0xFFFFFFFF, ((seed >> 32) ^ 0x53414D50) & 0xFFFFFFFF,
                         rid & M32, rid >> np.uint64(32), step & 0xFFFFFFFF, step >> 32)[0]


def uniform_f32(w0) -> np.ndarray:
    """The kernel's uniform, rounded as float32 rounds it: ((w0 >> 8) + 0.5f) * 2^-24.  For w0 >> 8 >= 2^23 the
    half is lost to rounding, so w0 >> 8 == 0xFFFFFF gives exactly 1.0: the range is (0, 1]."""
    k = (np.asarray(w0, dtype=np.uint32) >> np.uint32(8)).astype(np.float32)
    return (k + np.float32(0.5)) * np.float32(1.0 / 16777216.0)


def reference(logits, mask):
    """float64 log-softmax and cumulative mass of the masked logits, with the collector's guard (a row without a
    legal cell becomes all-legal) and the fill value as the logits' dtype stores it."""
    import torch
    eff = mask | ~mask.any(1, keepdim=True)
    fill = float(torch.tensor(FILL[str(logits.dtype).split(".")[-1]], dtype=logits.dtype))
    lsm = torch.log_softmax(logits.double().masked_fill(~eff, fill), dim=1)
    p = lsm.exp()
    return eff, lsm, p, p.cumsum(1)


def inverse_cdf(p, cdf, u):
    """First cell whose cumulative mass exceeds u; the last cell with mass when none does (u rounds up to 1)."""
    import torch
    A = p.shape[1]
    first = torch.searchsorted(cdf, u[:, None], right=True)[:, 0]
    last = (A - 1) - (p > 0).flip(1).to(torch.int8).argmax(1)
    return torch.where(first < A, first, last)


def make_rows(n: int, A: int, dtype, g):
    """Logits and masks in eight row kinds (row r is kind r % 8): random masks, masks of contiguous runs (about
    three lanes long, so whole lanes carry no mass), one legal cell, all legal, peaked (one cell ~1, the rest
    ~2^-20), uniform logits over runs, legal logits below the fill value (the masked cells get the mass, as in
    torch), and rows with no legal cell (the guard)."""
    import torch
    dev = g.device
    chunk = (A + 31) // 32
    kind = (torch.arange(n, device=dev) % 8)[:, None]
    z = torch.randn((n, A), generator=g, device=dev)
    bern = torch.rand((n, A), generator=g, device=dev) < 0.4
    seg = (torch.rand((n, A), generator=g, device=dev) < 1.0 / (3 * chunk)).long().cumsum(1)
    runs = (torch.rand((n, A + 1), generator=g, device=dev) < 0.5).gather(1, seg)
    hot = torch.zeros((n, A), dtype=torch.bool, device=dev)
    hot.scatter_(1, torch.randint(0, A, (n, 1), generator=g, device=dev), True)
    mask = torch.where(kind == 0, bern, runs)
    mask = torch.where(kind == 2, hot, mask)
    mask = torch.where(kind == 3, torch.ones_like(mask), mask)
    mask = torch.where(kind == 4, runs | hot, mask)
    mask = torch.where(kind == 7, torch.zeros_like(mask), mask)
    logits = 3.0 * z
    logits = torch.where(kind == 4, torch.where(hot, 0.0, math.log(2.0 ** -20) + 0.01 * z), logits)
    logits = torch.where(kind == 5, torch.zeros_like(z), logits)
    logits = torch.where(kind == 6, 2.0 * FILL[str(dtype).split(".")[-1]] + z, logits)
    return logits.to(dtype), mask


def test_numpy_philox_matches_oracle(oracle):
    rng = np.random.default_rng(5)
    words = rng.integers(0, 2 ** 32, size=(2000, 6), dtype=np.uint64)
    words[:500, 3:] = 0xFFFFFFFF                       # counters with high words set, and all-ones
    words[500:1000, 1] = 0
    keys, ctrs = words[:, :2], words[:, 2:]
    for (k0, k1), c in zip(keys, ctrs):
        got = philox4x32_10(int(k0), int(k1), *(int(x) for x in c))
        assert tuple(int(x) for x in got) == oracle.philox4x32_10((int(k0), int(k1)), tuple(int(x) for x in c))
    # vectorised over the counter, as the draw-by-draw test uses it
    key = (int(keys[0, 0]), int(keys[0, 1]))
    got = np.stack(philox4x32_10(*key, ctrs[:, 0], ctrs[:, 1], ctrs[:, 2], ctrs[:, 3]), 1)
    want = np.array([oracle.philox4x32_10(key, tuple(int(x) for x in c)) for c in ctrs], dtype=np.uint32)
    assert np.array_equal(got, want)


def _check_draws(torch, logits, mask_before, mask_after, a64, a32, logp, u64, label):
    """Assert every draw against the float64 inverse CDF; return (near-boundary fraction, tolerance-used fraction)."""
    n, A = logits.shape
    amin, amax = int(a64.min()), int(a64.max())
    assert 0 <= amin and amax < A, f"{label}: action outside [0, {A}): min {amin}, max {amax}"
    assert torch.equal(a64.to(torch.int32), a32)
    eff, lsm, p, cdf = reference(logits, mask_before)
    assert torch.equal(mask_after, eff), f"{label}: only rows without a legal cell may change the mask"
    exact = inverse_cdf(p, cdf, u64)
    u = u64[:, None]
    allowed = (p > 0) & (cdf - p <= u + BOUNDARY_TOL) & (cdf > u - BOUNDARY_TOL)
    ok = allowed.gather(1, a64[:, None])[:, 0]
    if not bool(ok.all()):
        r = int((~ok).nonzero()[0, 0])
        a, e = int(a64[r]), int(exact[r])
        raise AssertionError(f"{label}: {int((~ok).sum())} rows off the float64 inverse CDF; row {r}: action {a} "
                             f"(mass {float(p[r, a]):.3e}, cdf {float(cdf[r, a]):.9f}, legal {bool(eff[r, a])}), "
                             f"expected {e} (cdf {float(cdf[r, e]):.9f}), u {float(u64[r]):.9f}")
    want = lsm.gather(1, a64[:, None])[:, 0]
    err = (logp.double() - want).abs() - (LOGP_ATOL + LOGP_RTOL * want.abs())
    assert float(err.max()) <= 0, f"{label}: logp off float64 log_softmax by {float(err.max()):.3e} over tolerance"
    near = float((allowed.sum(1) > 1).double().mean())
    used = float((a64 != exact).double().mean())
    return near, used


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["float32", "float16", "bfloat16"])
@pytest.mark.parametrize("A", [1, 2, 31, 32, 33, 35, 81, 255, 256, 257, 480, 512, 513, 1000, 1024])
def test_draws_match_float64_inverse_cdf(dtype_name, A):
    """65,536 rows per case; non-zero row_id_base whose low word wraps inside the batch, a step_index >= 2^32 and a
    device epoch, so every draw also pins the counter layout (env sharding and graph replays rely on it)."""
    import torch
    from minesweeper_ppo_b200.rollout import masked_sample
    dt = getattr(torch, dtype_name)
    n = 65536
    seed = (0xA5A5 << 48) + 1000 * A + len(dtype_name)
    row_id_base, step_index, epoch = (3 << 32) - 1000, (1 << 32) + 77, 2
    g = torch.Generator(device="cuda").manual_seed(1000 * A + len(dtype_name))
    logits_all, mask_all = make_rows(n + 1, A, dt, g)      # one spare row: a stray read past row n-1 stays inside
    mask_before = mask_all.clone()
    logits, mask = logits_all[:n], mask_all[:n]
    a64, a32, logp = masked_sample(logits, mask, seed=seed, step_index=step_index, row_id_base=row_id_base,
                                   epoch=torch.tensor([epoch], dtype=torch.int32, device="cuda"))
    assert torch.equal(mask_all[n], mask_before[n])
    w0 = sampler_w0(seed, np.arange(n, dtype=np.uint64) + np.uint64(row_id_base), step_index, epoch)
    u64 = torch.from_numpy(uniform_f32(w0).astype(np.float64)).cuda()
    near, used = _check_draws(torch, logits, mask_before[:n], mask, a64, a32, logp, u64, f"{dtype_name} A={A}")
    print(f"\n{dtype_name} A={A}: near-boundary rows {near:.2e}, rows decided by the tolerance {used:.2e}")
    assert near <= NEAR_BOUNDARY_MAX and used <= DECIDED_MAX, (near, used)


@pytest.mark.gpu
@pytest.mark.parametrize("row_id_base,step_index,epoch", [
    (0, 0, None),
    ((1 << 32) - 30000, (5 << 32) + 3, 7),               # row id carries into the high word inside the batch
    ((0x7FFF << 48) + 12345, (0xFFFFFFFF << 32) + 9, 3),  # step high word + epoch wraps mod 2^32
])
def test_draw_keying_is_exact(row_id_base, step_index, epoch):
    """Zero logits over 1,024 legal cells make every float32 sum exact, so the action is floor(u * 1024) with no
    tolerance: a bit-for-bit check of the key and counter layout, the epoch and the uniform's rounding.  The same
    draws come back when the epoch is folded into the step and when the batch is split at a row boundary."""
    import torch
    from minesweeper_ppo_b200.rollout import masked_sample
    n, A, seed = 65536, 1024, 0x0123456789ABCDEF
    logits = torch.zeros((n, A), device="cuda")
    mask = torch.ones((n, A), dtype=torch.bool, device="cuda")
    ep = None if epoch is None else torch.tensor([epoch], dtype=torch.int32, device="cuda")
    a64, _, logp = masked_sample(logits, mask, seed=seed, step_index=step_index, row_id_base=row_id_base, epoch=ep)
    u = uniform_f32(sampler_w0(seed, np.arange(n, dtype=np.uint64) + np.uint64(row_id_base), step_index, epoch or 0))
    want = np.minimum(np.floor(u.astype(np.float64) * A), A - 1).astype(np.int64)
    got = a64.cpu().numpy()
    assert np.array_equal(got, want), f"{int((got != want).sum())} of {n} draws differ from the keyed reference"
    assert float((logp + math.log(A)).abs().max()) <= LOGP_ATOL
    folded = (step_index + ((epoch or 0) << 32)) & 0xFFFFFFFFFFFFFFFF
    b64, _, _ = masked_sample(logits, mask, seed=seed, step_index=folded, row_id_base=row_id_base)
    k = 12345
    c64, _, _ = masked_sample(logits[k:], mask[k:], seed=seed, step_index=step_index, row_id_base=row_id_base + k,
                              epoch=ep)
    assert torch.equal(a64, b64) and torch.equal(a64[k:], c64)


# Rows that hit the non-monotone lane scan.  Three legal cells carry the masses e, e and 1 (e = 0.7 * 2^-24) in
# consecutive lanes L, L+1, L+2; every other cell is masked.  The float32 scan then rounds 1 + e down to 1 in lane
# L+2 but 1 + 2e up to 1 + 2^-23 in a later, empty lane, which sits one ulp above the lanes before it (and, in some
# rows, above the total).  A uniform of 1 - 2^-23 or 1 lands in that gap.  e is far from both rounding thresholds
# (0.5 and 1 times 2^-24), so a few ulps of expf error change nothing.  Each case names the Philox word its counter
# must produce, the cell the float64 inverse CDF picks, and what the kernel returned before the owner lane had to
# carry mass (for the record: a masked cell, or an index >= A).
LANE_BOUNDARY_CASES = [
    # A, legal cells (mass e, e, 1), row_id_base, w0, float64 cell, previous kernel's action
    (35, (0, 2, 4), 12749683, 0xFFFFFE36, 4, 6),
    (35, (30, 32, 34), 1523505, 0xFFFFFF5A, 34, 36),
    (81, (72, 75, 78), 12749683, 0xFFFFFE36, 78, 81),          # 9x9 board, 3 cells a lane, lanes 27-31 past the row
    (300, (270, 280, 290), 1523505, 0xFFFFFF5A, 290, 300),    # 10 cells a lane (the 16-cell instance)
    (1000, (896, 928, 960), 12749683, 0xFFFFFE36, 960, 992),  # 32 cells a lane (the 32-cell instance)
]
LANE_SEED, LANE_STEP = 7, 3


@pytest.mark.gpu
@pytest.mark.parametrize("A,cells,row_id_base,w0,want,old", LANE_BOUNDARY_CASES,
                         ids=[f"A{c[0]}-{'past_row' if c[5] >= c[0] else 'masked'}" for c in LANE_BOUNDARY_CASES])
def test_lane_boundary_draw_stays_legal(A, cells, row_id_base, w0, want, old):
    import torch
    from minesweeper_ppo_b200.rollout import masked_sample
    assert int(sampler_w0(LANE_SEED, np.array([row_id_base], dtype=np.uint64), LANE_STEP)[0]) == w0
    e = math.log(0.7 * 2.0 ** -24)
    # the row is an n = 1 view of a 4-row allocation, so a read past the row stays inside it
    logits = torch.zeros((4, A), device="cuda")
    mask = torch.zeros((4, A), dtype=torch.bool, device="cuda")
    for c, x in zip(cells, (e, e, 0.0)):
        logits[0, c], mask[0, c] = x, True
    mask_before = mask.clone()
    a64, a32, logp = masked_sample(logits[:1], mask[:1], seed=LANE_SEED, step_index=LANE_STEP,
                                   row_id_base=row_id_base)
    action, lp = int(a64[0]), float(logp[0])
    was = f"(the selection without the owner-has-mass rule returned {old})"
    assert 0 <= action < A, f"action {action} outside the row (A = {A}) {was}"
    assert bool(mask_before[0, action]), f"action {action} is masked, legal cells {cells} {was}"
    assert int(a32[0]) == action and torch.equal(mask, mask_before)
    _, lsm, p, cdf = reference(logits[:1], mask_before[:1])
    u64 = torch.tensor([float(uniform_f32(np.uint32(w0)))], dtype=torch.float64, device="cuda")
    assert int(inverse_cdf(p, cdf, u64)[0]) == want == action
    assert math.isfinite(lp) and abs(lp - float(lsm[0, action])) <= LOGP_ATOL
