#!/usr/bin/env python
"""Benchmark of the rollout hot path (BASELINE.json metric: env steps/s, 16x16x40).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...    # CPU arm (oracle port, all host threads)
    torchrun --nproc-per-node N bench.py --gpus N ...              # one rank per GPU, env shards, weak scaling

Workload (config.workload = "C2"): BASELINE.json configs[1] -- 16x16x40, 65,536 envs per GPU,
uniformly random VALID action per env per step (drawn on device), auto-reset on.
A "step" is one VecMinesweeper.step over all envs of the rank = ONE fused launch (synthetic action
draw, board generation on first clicks, flood fill, win/loss, reward, auto-reset, obs + mask encode
written into a ring of rollout-buffer slots).

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "env_steps_per_s"
UNIT = "env-steps/s"
H, W, MINES = 16, 16, 40
ENVS_PER_GPU = 65536
# SURVEY 8(d): algorithmic bytes per env-step at the boundary (fp32 reference layout):
# obs 40*HW + mask HW + reward 4 + done 1 + action 4
BYTES_PER_STEP = 41 * H * W + 9          # 10,505 B
WORKLOAD = "C2"
VALID_ONLY = True
# Workload setup, both arms: reset() starts every env's first episode at the same instant, so the first ~20 steps are
# not random play in steady state (every env opens its first region together, then the first wave of losses ...).
# PRE_ROLL untimed env steps after reset() bring the batch to the stationary mix of episode phases (episodes last
# ~5.6 steps under random play) before the W warm-up and K timed steps.
PRE_ROLL = 32
# --dump-outputs writes a fixed, seeded sample of the envs (all their outputs), at most this many and DUMP_BYTES in all
DUMP_ENVS = 4096
DUMP_BYTES = 56 << 20


def set_workload(name: str, envs):
    """C2 = BASELINE.json configs[1] (the bench line); C4 = configs[3], Expert 16x30x99 boards,
    4,194,304 envs sharded over 8 GPUs = 524,288 per GPU (a parity-test size, offered for sweeps)."""
    global H, W, MINES, ENVS_PER_GPU, BYTES_PER_STEP, WORKLOAD
    if name == "C4":
        H, W, MINES, ENVS_PER_GPU = 16, 30, 99, 524288
    elif name != "C2":
        raise SystemExit(f"unknown workload {name}")
    WORKLOAD = name
    if envs:
        ENVS_PER_GPU = int(envs)
    BYTES_PER_STEP = 41 * H * W + 9


def env_cfg(mod):
    return mod.EnvConfig(H=H, W=W, mine_count=MINES, guarantee_safe_neighborhood=True, step_penalty=1e-4)


def bench_config(world: int) -> dict:
    """The workload both arms run (identical dict in the CUDA arm and in --impl reference)."""
    return {
        "workload": WORKLOAD, "board": f"{H}x{W}x{MINES}", "envs_per_gpu": ENVS_PER_GPU,
        "envs_total": ENVS_PER_GPU * world,
        "actions": ("uniform random valid cell" if VALID_ONLY else "uniform random cell (series B, no-op clicks included)")
                   + " per env per step",
        "auto_reset": True, "pre_roll_steps": PRE_ROLL, "obs_layout": f"fp32 [N,10,{H},{W}] + bool mask [N,{H * W}] (reference layout)",
        "l2": f"each step writes {BYTES_PER_STEP * ENVS_PER_GPU / 1e6:.0f} MB of obs/mask (>> 126 MB L2), no explicit flush",
        "parallelism": f"env shards, {world} rank(s), no data-path collective",
    }


def numba_reference_baseline(quick: bool = False):
    """BASELINE.md section 4 (i)/(ii): the REAL reference env (Python + numba, baseline/_ref) timed on this
    box's host cores by tools/numba_reference_bench.py in a fresh interpreter."""
    import subprocess
    cmd = [sys.executable, os.path.join(ROOT, "tools", "numba_reference_bench.py")] + (["--quick"] if quick else [])
    try:
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600,
                           env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        if r.returncode != 0 or not lines:
            return {"unavailable": f"numba_reference_bench rc={r.returncode}: {r.stderr.strip()[-300:]}"}
        return json.loads(lines[-1])
    except Exception as e:  # pragma: no cover
        return {"unavailable": repr(e)}


# ----------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}

    def __init__(self, torch, dev_index: int, period_s: float = 0.01):
        super().__init__(daemon=True)
        self.period, self.samples, self.reasons, self.sm_max, self.err = period_s, [], set(), None, None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            p = torch.cuda.get_device_properties(dev_index)
            try:
                bus = "%08x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(dev_index)
            self.nv = pynvml
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # pragma: no cover
            self.nv, self.err = None, repr(e)

    def sample_once(self):
        nv = self.nv
        self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
        for bit, name in self.REASONS.items():
            if r & bit:
                self.reasons.add(name)

    def run(self):
        # The first sample is taken one period AFTER the start: an NVML query issued while the main thread is still
        # queueing the first launches contends with it for the driver and starves the GPU between launches (20 timed
        # launches measured 108.6 us per step with a sample at t = 0, 103.6 us steady state in tools/warm_probe.py).
        # A region shorter than one period gets its sample from finish(), which runs while the GPU is still busy.
        if self.nv is None:
            return
        while not self._stop_evt.wait(self.period):
            try:
                self.sample_once()
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
                break

    def finish(self):
        """Call while the GPU is still busy with the timed region (before the final synchronize), so
        even a very short region gets at least one sample under load."""
        if self.nv is not None and self.err is None:
            try:
                self.sample_once()
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
        self._stop_evt.set()
        self.join(timeout=2)
        out = {"sm_mhz": (float(np.median(self.samples)) if self.samples else None), "sm_max_mhz": self.sm_max,
               "reasons": sorted(self.reasons), "samples": len(self.samples)}
        if self.err:
            out["error"] = self.err
        return out


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled_traffic():
    """Per-launch DRAM bytes of the env step kernel from the committed ncu capture (profiles/)."""
    try:
        with open(os.path.join(ROOT, "profiles", "env_step_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


# ----------------------------------------------------------------------------- CPU arm
def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_env_steps_per_s(n_envs: int, steps: int, warmup: int, threads: int):
    """Oracle port of VecMinesweeper.step on `threads` host threads; timing around step only
    (BASELINE.md section 4), random valid actions prepared outside the timed region."""
    from oracle import oracle as O
    cfg = O.OracleEnvConfig(H=H, W=W, mine_count=MINES, guarantee_safe_neighborhood=True, step_penalty=1e-4)
    vec = O.OracleVecEnv(n_envs, cfg, seed=0, nthreads=threads, reuse_out=True)
    rng = np.random.default_rng(1)
    mask = vec.reset()["action_mask"]
    total = 0.0
    per_step = []
    warmup += PRE_ROLL                     # untimed: pre-roll to the stationary episode mix, then the warm-up steps
    for t in range(warmup + steps):
        s = rng.random(mask.shape, dtype=np.float32)
        s[~mask] = -1.0
        a = s.argmax(1)
        t0 = time.perf_counter()
        b, _, _, _ = vec.step(a, tensor_infos=True)
        dt = time.perf_counter() - t0
        mask = b["action_mask"]
        if t >= warmup:
            total += dt
            per_step.append(dt)
    return n_envs * steps / total, total, per_step


def run_reference_arm(args, rank: int, world: int):
    if rank != 0:
        return
    threads = host_threads()
    # calibrate a bounded sample so warmup+steps finish in ~2 minutes
    rate, _, _ = cpu_env_steps_per_s(4096, 3, 1, threads)
    budget_s = 100.0
    n = int(max(1024, min(ENVS_PER_GPU, rate * budget_s / max(1, args.steps + args.warmup + PRE_ROLL))))
    n = 1 << (n.bit_length() - 1)
    value, total, per_step = cpu_env_steps_per_s(n, args.steps, args.warmup, threads)
    sample = f"{n} envs x {args.steps} steps, {H}x{W}x{MINES} random valid actions, oracle/msw_oracle.c (C port), {threads} threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": bench_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "envs_sampled": n, "reference_numba": numba_reference_baseline()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "value = the C restatement of the reference's algorithm (oracle/msw_oracle.c) on all host threads -- "
                "the FASTEST CPU implementation available, so the GPU/CPU ratio is conservative; the unmodified "
                "Python+numba reference timed on the same cores is cpu_baseline.reference_numba (one core as "
                "shipped, and a P-process fan-out)",
    }
    emit_json(line)


# ----------------------------------------------------------------------------- CUDA arm
def dump_outputs(torch, out_dir, step_out, actions):
    """--dump-outputs: what one step returned to its caller (obs, action mask, rewards, dones and the actions the
    built-in policy drew) for a fixed, seeded sample of the envs, as float32 .npy files; env_index.npy (float64)
    names the sampled envs."""
    n = actions.shape[0]
    per_env = 4 * (step_out.obs[0].numel() + step_out.action_mask[0].numel() + 3) + 8
    rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_ENVS, DUMP_BYTES // per_env), replace=False))
    idx = torch.from_numpy(rows).to(actions.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), rows.astype(np.float64))
    for name, t in (("obs", step_out.obs), ("action_mask", step_out.action_mask), ("rewards", step_out.rewards),
                    ("dones", step_out.dones), ("actions", actions)):
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(0, idx).float().cpu().numpy())


def time_env_steps(torch, m, dev, rank, world, barrier, board, n_envs, K, Wm, ring, valid_only=True, dump_dir=None):
    """The device-timed leg for one board/env-count: PRE_ROLL + W untimed and K timed fused step launches (built-in
    synthetic policy), CUDA events around the K launches only; then a separate replay that measures the per-launch
    kernel time for the roofline (back to back between one event pair, and with an event pair around each launch).
    With `dump_dir`, the outputs of the last timed step are written there (dump_outputs) before the replay.
    Returns (ms of the K timed launches, kernel ms back to back, clocks, kernel ms bracketed)."""
    h, w, mines = board
    cfg = m.EnvConfig(H=h, W=w, mine_count=mines, guarantee_safe_neighborhood=True, step_penalty=1e-4)
    vec = m.VecMinesweeper(n_envs, cfg, seed=0, api="torch", env_id_base=rank * n_envs)
    slots = [m.StepOut(obs=torch.empty((n_envs, 10, h, w), dtype=torch.float32, device=dev),
                       action_mask=torch.empty((n_envs, h * w), dtype=torch.bool, device=dev),
                       rewards=torch.empty((n_envs,), dtype=torch.float32, device=dev),
                       dones=torch.empty((n_envs,), dtype=torch.bool, device=dev)) for _ in range(ring)]
    scratch = torch.empty((n_envs,), dtype=torch.int32, device=dev)
    vec.reset(out=slots[0])
    for t in range(PRE_ROLL):                                    # workload setup: stationary mix of episode phases
        vec.step_random(t, valid_only=valid_only, out=slots[t % ring], actions_out=scratch)
    Wm = Wm + PRE_ROLL                                           # step indices continue after the pre-roll
    for t in range(PRE_ROLL, Wm):
        vec.step_random(t, valid_only=valid_only, out=slots[t % ring], actions_out=scratch)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(torch, dev.index)
    barrier()
    sampler.start()
    ev0.record()
    for t in range(K):
        vec.step_random(Wm + t, valid_only=valid_only, out=slots[t % ring], actions_out=scratch)   # policy + step: one launch
    ev1.record()
    clocks = sampler.finish()          # sampled while the last launches are still executing
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    if dump_dir is not None:
        dump_outputs(torch, dump_dir, slots[(K - 1) % ring], scratch)
    # Per-launch kernel time for the roofline, from a separate replay after the timed region: Kk launches back to back
    # between ONE event pair (launches of one stream do not overlap, so elapsed / Kk bounds the mean kernel duration
    # from above), after 5 launches that absorb the restart after the barrier.  An event pair around EACH launch adds
    # ~2 us of front-end gap to every launch (`bracketed`, kept for reference).
    Kk = min(64, max(8, K))
    for t in range(5):
        vec.step_random(Wm + K + t, valid_only=valid_only, out=slots[t % ring], actions_out=scratch)
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for t in range(Kk):
        vec.step_random(Wm + K + 5 + t, valid_only=valid_only, out=slots[t % ring], actions_out=scratch)
    r1.record()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(Kk)]
    for t in range(Kk):
        kev[t][0].record()
        vec.step_random(Wm + K + 5 + Kk + t, valid_only=valid_only, out=slots[t % ring], actions_out=scratch)
        kev[t][1].record()
    barrier()
    ms_kernel = r0.elapsed_time(r1) / Kk
    ms_kernel_bracketed = float(np.mean([x.elapsed_time(y) for x, y in kev]))
    del vec, slots
    return ms_total, ms_kernel, clocks, ms_kernel_bracketed


def record_actions(torch, m, dev, rank, board, n_envs, steps, valid_only=True):
    """int32 [steps, n_envs]: the built-in synthetic policy's actions for `steps` steps after reset() + PRE_ROLL
    steps (the trajectory the e2e legs replay through msw_step_host)."""
    h, w, mines = board
    cfg = m.EnvConfig(H=h, W=w, mine_count=mines, guarantee_safe_neighborhood=True, step_penalty=1e-4)
    vec = m.VecMinesweeper(n_envs, cfg, seed=0, api="torch", env_id_base=rank * n_envs)
    out = m.StepOut(obs=torch.empty((n_envs, 10, h, w), dtype=torch.float32, device=dev),
                    action_mask=torch.empty((n_envs, h * w), dtype=torch.bool, device=dev),
                    rewards=torch.empty((n_envs,), dtype=torch.float32, device=dev),
                    dones=torch.empty((n_envs,), dtype=torch.bool, device=dev))
    log = torch.empty((steps, n_envs), dtype=torch.int32, device=dev)
    scratch = torch.empty((n_envs,), dtype=torch.int32, device=dev)
    vec.reset(out=out)
    for t in range(PRE_ROLL):
        vec.step_random(t, valid_only=valid_only, out=out, actions_out=scratch)
    for t in range(steps):
        vec.step_random(PRE_ROLL + t, valid_only=valid_only, out=out, actions_out=log[t])
    torch.cuda.synchronize()
    return log


def run_cuda_arm(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist
    import minesweeper_ppo_b200 as m

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    N = ENVS_PER_GPU
    K, Wm = args.steps, args.warmup
    cfg = env_cfg(m)
    ring = 4 if WORKLOAD == "C2" else 2        # rollout-buffer slots the obs/mask stream into

    def make_env():
        return m.VecMinesweeper(N, cfg, seed=0, api="torch", env_id_base=rank * N)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather(x: float):
        if world == 1:
            return [x]
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    Ke = min(K, 400)                           # steps replayed by the e2e legs
    ms_total, ms_kernel, clocks, ms_kernel_bracketed = time_env_steps(torch, m, dev, rank, world, barrier, (H, W, MINES),
                                                                      N, K, Wm, ring, VALID_ONLY,
                                                                      args.dump_outputs if rank == 0 else None)
    # The actions the e2e legs replay are recorded in a separate untimed pass over the same deterministic trajectory
    # (recording inside the timed launches costs 3 us per launch: 65,536 four-byte stores into a row of device memory
    # that is cold every step, against a scratch row that stays in L2).
    actions_log = record_actions(torch, m, dev, rank, (H, W, MINES), N, Wm + Ke, VALID_ONLY)
    episodes = None

    # -- e2e: same workload through the host-buffer C-ABI call (msw_step_host): per step, this
    # step's actions come from pinned host memory (H2D) and rewards+dones go back to pinned host
    # memory (D2H); obs/mask land in device memory where the policy consumes them.
    # The recorded actions live in ONE pinned allocation, a different 256 KB row per step.  How long a 256 KB DMA takes
    # depends on where the piece of pinned memory lies physically (17 us or 25-36 us, profiles/r02aj_pinned_probe.txt);
    # the last three rows of the unpadded allocation were slow ones (+45 us on steps 17-19 of 20 in
    # profiles/r02ah_bench_e2e_tail_rows.json), the middle rows of a padded allocation have been uniformly fast in every
    # run since.  Hence 2 MB of padding on either side of the rows that are used.
    pad = max(1, (2 << 20) // (4 * N))
    acts_pinned = torch.empty((Wm + Ke + 2 * pad, N), dtype=torch.int32).pin_memory()
    acts_host = acts_pinned[pad:pad + Wm + Ke]
    acts_host.copy_(actions_log[: Wm + Ke])
    torch.cuda.synchronize()
    del actions_log
    torch.cuda.empty_cache()

    step_ms = {}
    exp_threads = max(1, host_threads() // world)      # host threads of the NumPy-result expansion: the box's cores / ranks

    def run_host(copy_obs: bool, steps: int, delta: bool = True):
        v = make_env()
        v.host_delta = delta
        v.reset()
        scratch = torch.empty((N,), dtype=torch.int32, device=dev)
        pre = m.StepOut(obs=torch.empty((N, 10, H, W), dtype=torch.float32, device=dev),
                        action_mask=torch.empty((N, H * W), dtype=torch.bool, device=dev),
                        rewards=torch.empty((N,), dtype=torch.float32, device=dev),
                        dones=torch.empty((N,), dtype=torch.bool, device=dev))
        for t in range(PRE_ROLL):              # the same untimed pre-roll as the device-timed leg (same trajectory)
            v.step_random(t, valid_only=VALID_ONLY, out=pre, actions_out=scratch)
        del pre, scratch
        pin = None
        done_count = 0
        for t in range(Wm):                    # warm up exactly as the timed loop runs: the previous result stays
            pin = v.step_host(acts_host[t], copy_obs=copy_obs, copy_infos=False, threads=exp_threads)   # referenced and
            done_count += int(np.count_nonzero(pin["done"].numpy()))                                     # the host reads it
        rows = [acts_host[Wm + t] for t in range(steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); e1.record()               # events are created lazily at their first record: not inside the timed region
        gc.disable()                           # as timeit does: no cyclic-GC pass inside a 3 ms timed region
        barrier()
        t0 = time.perf_counter()
        e0.record()
        done_count = 0
        stamps = [t0]
        for a in rows:
            pin = v.step_host(a, copy_obs=copy_obs, copy_infos=False, threads=exp_threads)
            done_count += int(np.count_nonzero(pin["done"].numpy()))   # the host really reads the result
            stamps.append(time.perf_counter())
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        gc.enable()
        step_ms[(copy_obs, delta)] = [round(1e3 * (b - a), 4) for a, b in zip(stamps[:-1], stamps[1:])][:64]
        return max(e0.elapsed_time(e1) / 1e3, wall), wall, done_count

    if args.no_e2e:
        Kh = Kf = 1
        e2e_s, e2e_full_s, e2e_rewrite_s, episodes = float("inf"), float("inf"), float("inf"), None
    else:
        e2e_s, e2e_wall, episodes = run_host(False, Ke)
        Kh = Ke
        e2e_full_s, _, _ = run_host(True, Kh)
        Kf = min(Ke, 12)
        e2e_rewrite_s, _, _ = run_host(True, Kf, delta=False)

    ms_total_max = reduce_max(ms_total)
    e2e_s_max = reduce_max(e2e_s)
    e2e_full_max = reduce_max(e2e_full_s)
    e2e_rewrite_max = reduce_max(e2e_rewrite_s)
    # The timed region holds nothing but K launches of the step kernel, so the kernel's average launch duration over
    # the timed region is ms_total / K (per rank; the slowest rank bounds the roofline figure).
    kernel_ms_ranks = gather(ms_total / K)
    ms_kernel_max = max(kernel_ms_ranks)
    replay_ms_max = reduce_max(ms_kernel)
    del acts_host, acts_pinned
    torch.cuda.empty_cache()

    gae_info = None if args.no_gae else bench_gae(torch, m, dev)
    roll_info = None if args.no_rollout else bench_rollout(torch, m, dev, rank, world, reduce_max)
    c4_info = None if (args.no_c4 or WORKLOAD != "C2") else bench_c4(torch, m, dev, rank, world, barrier, reduce_max, gather)
    c5_info = None if args.no_train else bench_train_c5(torch, m, dev, rank, world)

    if rank != 0:
        return
    total_envs = N * world
    value = total_envs * K / (ms_total_max / 1e3)
    peak, peak_src = measured_peak_gbs()
    achieved = BYTES_PER_STEP * N / (ms_kernel_max / 1e3) / 1e9
    traffic = profiled_traffic() if (WORKLOAD == "C2" and N == 65536) else None
    config = bench_config(world)
    config["action_source"] = ("drawn inside the step launch (msw_step rand_mode; bit-identical to msw_random_actions); "
                               f"obs/mask stream into a ring of {ring} rollout-buffer slots")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_total_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": config,
        "roofline": {
            "bound": "hbm", "kernel": f"msw::env_kernel<MODE_STEP,{W},{H * W}>", "achieved": achieved, "peak": peak,
            "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
            "peak_note": "hbm_gbs is a read+write copy; this kernel only writes, and write-only streams reach 6.9-7.0 TB/s "
                         "on this part (profiles/r01_store_probe2.txt), so a fraction near or slightly above 1.0 of the "
                         "copy peak is the practical ceiling",
            "algorithmic_bytes_per_launch": BYTES_PER_STEP * N, "kernel_ms": ms_kernel_max,
            "kernel_ms_per_rank": kernel_ms_ranks,
            "kernel_ms_how": "the timed region holds only the K launches of this kernel: CUDA-event time of the region / K, "
                             "per rank, max over ranks",
            "kernel_ms_replay": replay_ms_max,
            "kernel_ms_replay_how": "separate replay after the timed region and 5 more launches: min(64, K) launches back to "
                                    "back between one CUDA-event pair, elapsed / count (the first launches after a "
                                    "synchronize run ~4 us slower, so a 20-launch timed region sits between this figure and "
                                    "the bracketed one); max over ranks",
            "kernel_ms_bracketed": ms_kernel_bracketed,
            "kernel_ms_bracketed_how": "the same replay with an event pair around EACH launch (adds ~2 us of front-end "
                                       "gap per launch); rank 0",
            "traffic": (traffic or {}).get("dram_bytes_per_launch"),
            "traffic_source": (traffic or {}).get("source"),
        },
        "e2e": {
            "value": total_envs * Ke / e2e_s_max, "unit": UNIT, "steps": Ke,
            "h2d_bytes_per_step": 4 * N, "d2h_bytes_per_step": 5 * N,
            "call": "msw_step_host via VecMinesweeper.step_host(copy_obs=False): pinned int32 actions in, "
                    "pinned reward f32 + done bool out, stream-synchronised every step; obs/mask stay in HBM "
                    "for the policy (the reference copies obs host->device at this point, train_rl.py:198-199)",
            "step_ms": step_ms.get((False, True)),
        },
        "e2e_host_obs": {
            "value": total_envs * Kh / e2e_full_max, "unit": UNIT, "steps": Kh,
            "h2d_bytes_per_step": 4 * N, "d2h_bytes_per_step": host_obs_d2h_bytes(m, N),
            "call": "same call with copy_obs=True: the full reference-shaped NumPy result (obs fp32 [N,10,H,W] + mask + "
                    "reward + done) in host memory every step.  The planes do not cross PCIe: msw_step_host copies the "
                    "packed mine + revealed bitboards (64 B/env, in slices that overlap the expansion) and expands them on the host threads (msw_host_expand.cpp).  The "
                    "result arrays are recycled (two sets alternate here, as in any loop that keeps the previous batch) "
                    "and each carries a shadow of the bit planes it holds, so only the cache lines that changed since "
                    "the set was last filled are rewritten (non-temporal stores)",
            "full_rewrite": {"value": total_envs * Kf / e2e_rewrite_max, "steps": Kf,
                             "note": f"host_delta=False: every byte of obs/mask rewritten each step "
                                     f"({(41 * H * W) * N / 1e6:.0f} MB, bound by host store bandwidth)"},
            "host_threads_per_rank": exp_threads,
            "step_ms": step_ms.get((True, True)),
        },
        "gpu_launches": K,
        "gae": gae_info,
        "rollout": roll_info,
        "c4": c4_info,
        "train_c5": c5_info,
        "clocks": clocks,
        "episodes_finished_in_e2e": episodes,
    }
    if world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        rate, _, _ = cpu_env_steps_per_s(4096, 3, 1, threads)
        n_c = ENVS_PER_GPU
        steps_c = int(max(8, min(4000, rate * 12.0 / n_c)))      # about 10-15 s of CPU work
        v_c, total_c, _ = cpu_env_steps_per_s(n_c, steps_c, 2, threads)
        line["cpu_baseline"] = {
            "value": v_c, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n_c} envs x {steps_c} steps of the same workload on the host ({total_c:.1f} s), "
                      "oracle/msw_oracle.c (C restatement of env.py/env_numba.py) on all host threads",
            "reference_numba": numba_reference_baseline(),
        }
    emit_json(line)


def host_obs_d2h_bytes(m, n_envs: int) -> int:
    """Bytes msw_step_host moves device->host per step when the caller wants obs+mask on the host."""
    f = getattr(m.VecMinesweeper, "host_obs_d2h_bytes", None)
    return int(f(H, W, n_envs)) if f else (40 * H * W + H * W + 5) * n_envs


def bench_c4(torch, m, dev, rank, world, barrier, reduce_max, gather):
    """BASELINE.json configs[3] (C4): Expert boards (H=16, W=30, 99 mines), 524,288 envs per GPU
    (= 4,194,304 over 8 GPUs), env-only random valid actions; roofline at 19,689 B per env-step."""
    h, w, mines, n = 16, 30, 99, 524288
    K, Wm = 12, 3
    bps = 41 * h * w + 9
    ms_total, ms_kernel, _, _ = time_env_steps(torch, m, dev, rank, world, barrier, (h, w, mines), n, K, Wm, 2)
    torch.cuda.empty_cache()
    ms_max = reduce_max(ms_total)
    kr = gather(ms_total / K)                 # the timed region holds only the K launches of the step kernel
    peak, _ = measured_peak_gbs()
    ach = bps * n / (max(kr) / 1e3) / 1e9
    return {"workload": "C4", "board": f"{h}x{w}x{mines}", "envs_per_gpu": n, "envs_total": n * world, "steps": K,
            "env_steps_per_s": n * world * K / (ms_max / 1e3), "ms_per_step": ms_max / K,
            "algorithmic_bytes_per_env_step": bps, "kernel_ms": max(kr), "kernel_ms_per_rank": kr,
            "achieved_gbs": ach, "frac_of_hbm_peak": ach / peak,
            "l2": f"each step writes {bps * n / 1e9:.1f} GB into a ring of 2 slots, no explicit flush"}


def bench_train_c5(torch, m, dev, rank, world):
    """BASELINE.json configs[4] (C5): the full PPO loop of the medium config (16x16x40, 96x5 residual CNN),
    2,048 envs x 64 steps per GPU, env shards per GPU, ONE NCCL all-reduce of the flat gradient per
    optimizer step; 1 warm-up + 2 timed updates."""
    from minesweeper_ppo_b200 import train as T
    r = T.train(os.path.join(ROOT, "configs", "medium_16x16x40.yaml"), updates=3, envs_per_gpu=2048, steps=64, seed=0,
                log=lambda s: None, time_allreduce=True)
    torch.cuda.empty_cache()
    return r if rank == 0 else None


def bench_gae(torch, m, dev):
    """msw_gae at C3 size (T=128, N=8192; BASELINE.md section 4 inputs), CUDA-event timed."""
    T, N = 128, 8192
    g = torch.Generator(device=dev).manual_seed(0)
    buf = m.RolloutBuffer(N, T, (1, 1, 1), 1, dev)
    consts = torch.tensor([-1e-4, -1.0 - 1e-4, 1.0 - 1e-4], dtype=torch.float64).float().to(dev)
    dones = torch.rand((T * N,), device=dev, generator=g) < 0.15
    buf.dones.copy_(dones)
    buf.rewards.copy_(torch.where(dones, consts[torch.randint(1, 3, (T * N,), device=dev, generator=g)], consts[0]))
    buf.values.copy_(0.5 * torch.randn((T * N,), device=dev, generator=g))
    last = 0.5 * torch.randn((N,), device=dev, generator=g)
    flush = torch.empty(1 << 30, dtype=torch.uint8, device=dev)   # 1 GB >> L2; also keeps the host ahead of the GPU
    cold = []
    for i in range(13):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        buf.compute_gae(last, 0.995, 0.95)
        b.record()
        torch.cuda.synchronize()
        if i >= 3:
            cold.append(a.elapsed_time(b))
    def graph_us(b_, last_, reps=20):
        """Device time per launch with the host out of the way: `reps` launches captured in one CUDA graph."""
        gr, st = torch.cuda.CUDAGraph(), torch.cuda.Stream()
        with torch.cuda.stream(st):
            b_.compute_gae(last_, 0.995, 0.95)
            torch.cuda.synchronize()
            with torch.cuda.graph(gr, stream=st):
                for _ in range(reps):
                    b_.compute_gae(last_, 0.995, 0.95)
        gr.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); gr.replay(); e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / reps

    warm_ms = graph_us(buf, last) / 1e3
    # the same kernel where it is bandwidth- rather than latency-bound: 64x the columns (1.14 GB of traffic >> L2)
    NL = 64 * N
    big = m.RolloutBuffer(NL, T, (1, 1, 1), 1, dev)
    big.dones.copy_(torch.rand((T * NL,), device=dev, generator=g) < 0.15)
    big.rewards.copy_(torch.where(big.dones, consts[1], consts[0]))
    big.values.copy_(0.5 * torch.randn((T * NL,), device=dev, generator=g))
    big_us = graph_us(big, 0.5 * torch.randn((NL,), device=dev, generator=g), reps=5)
    big_bytes = 17 * T * NL + 4 * NL
    del big
    ms = float(np.median(cold))
    nbytes = 17 * T * N + 4 * N
    peak, _ = measured_peak_gbs()
    # CPU baseline (BASELINE.md section 4.3): the reference's loop (buffers.py:85-94) on CPU tensors
    r_c, v_c, d_c, lv_c = (x.cpu() for x in (buf.rewards.view(T, N), buf.values.view(T, N), buf.dones.view(T, N), last))
    cpu_ms = []
    for _ in range(3):
        t0 = time.perf_counter()
        adv_c = torch.zeros_like(v_c)
        last_adv = torch.zeros((N,), dtype=torch.float32)
        for t in reversed(range(T)):
            nv = lv_c if t == T - 1 else v_c[t + 1]
            nnt = 1.0 - d_c[t].float()
            delta = r_c[t] + 0.995 * nv * nnt - v_c[t]
            last_adv = delta + 0.995 * 0.95 * nnt * last_adv
            adv_c[t] = last_adv
        ret_c = adv_c + v_c
        cpu_ms.append((time.perf_counter() - t0) * 1e3)
    same = bool(torch.equal(adv_c, buf.advantages.view(T, N).cpu()) and torch.equal(ret_c, buf.returns.view(T, N).cpu()))
    return {"T": T, "N": N, "kernel_us": ms * 1e3,
            "cpu_reference_loop_ms": float(np.median(cpu_ms)), "cpu_threads": torch.get_num_threads(),
            "bit_identical_to_cpu_loop": same, "algorithmic_bytes": nbytes, "achieved_gbs": nbytes / ms / 1e6,
            "frac_of_hbm_peak": nbytes / ms / 1e6 / peak, "l2": "1 GB flush write before every timed launch (cold)",
            "back_to_back_us": warm_ms * 1e3,
            "large": {"T": T, "N": NL, "kernel_us": big_us, "algorithmic_bytes": big_bytes,
                      "achieved_gbs": big_bytes / big_us / 1e3, "frac_of_hbm_peak": big_bytes / big_us / 1e3 / peak},
            "note": "cold = inputs in HBM, CUDA events around one launch (about 3 us of that is event/launch gap: ncu "
                    "shows 11 us); back_to_back = 20 launches replayed from one CUDA graph (17.9 MB working set stays "
                    "in L2, as it does right after a rollout); at C3 size the kernel is latency-bound (8,192 chains "
                    "of 128 dependent steps, four 9 KB slices per CTA through the ring); `large` is the same kernel at 64x the columns, "
                    "where it is HBM-bound"}


def bench_rollout(torch, m, dev, rank, world, reduce_max):
    """BASELINE.json configs[2] (C3): PPO rollout + GAE, medium residual CNN (96 ch x 5 blocks,
    random init), fp16 autocast semantics, fused masked sampler, 8,192 envs x 128 steps per GPU,
    aux maps on.  Reported twice: with the fused GroupNorm forward (msw_gn_act between cuDNN convs)
    and with the unchanged eager PyTorch module."""
    N, T = 8192, 128
    cfg = env_cfg(m)

    def run(fused: bool, timed: int):
        torch.manual_seed(0)
        vec = m.VecMinesweeper(N, cfg, seed=0, api="torch", env_id_base=rank * N)
        model = m.build_model("cnn_residual", obs_shape=(10, H, W),
                              model_cfg=dict(stem_channels=96, blocks=5, dropout=0.05, value_hidden=256)).to(dev)
        col = m.RolloutCollector(vec, T, aux_maps=True, fused=fused)
        times, episodes = [], 0
        for i in range(1 + timed):
            torch.cuda.synchronize()
            a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            a.record()
            buf, aux = col.collect(model)
            b.record()
            buf.compute_gae(aux["last_values"], 0.995, 0.95)
            c.record()
            torch.cuda.synchronize()
            if i >= 1:
                times.append((a.elapsed_time(b), b.elapsed_time(c)))
            episodes = int(buf.dones.sum())
        del col, vec, model, buf
        torch.cuda.empty_cache()
        ms_roll = float(np.mean([t[0] for t in times]))
        ms_gae = float(np.mean([t[1] for t in times]))
        return ms_roll, ms_gae, reduce_max(ms_roll + ms_gae), episodes

    ms_roll, ms_gae, ms, episodes = run(True, 2)
    s_roll, s_gae, s_ms, _ = run(False, 1)
    flops = 0.44e9 * N * (T + 1)                      # SURVEY section 2: ~0.44 GFLOP / board / forward
    return {"workload": "C3", "frames_per_s": world * N * T / (ms / 1e3), "envs_per_gpu": N, "steps": T,
            "ms_rollout": ms_roll, "ms_gae": ms_gae,
            "forward": "stem + trunk 3x3 convs on tcgen05 with GroupNorm / ReLU / Dropout2d / fp32 residual add fused into the epilogue (msw_conv3x3_gn, obs packed by msw_pack_obs16) + fused per-cell heads on tcgen05 (msw_cell_heads); no cuDNN on the path",
            "model": "cnn_residual 96x5 (950,947 params), random init, train mode (dropout on, as the reference)",
            "model_tflops_est": flops / (ms_roll / 1e3) / 1e12, "episodes_in_buffer": episodes,
            "stock_module_forward": {"frames_per_s": world * N * T / (s_ms / 1e3), "ms_rollout": s_roll,
                                     "forward": "unchanged eager PyTorch module under fp16 autocast"}}


class _QuietStdout:
    """Route fd 1 to stderr while the benchmark runs (NCCL / library banners must not precede the
    JSON line on stdout); `emit` writes to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self._real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text: str):
        sys.stdout.flush()
        os.write(self._real, (text + "\n").encode())

    def close(self):
        sys.stdout.flush()
        os.dup2(self._real, 1)
        os.close(self._real)


OUT = None


def emit_json(line: dict):
    text = json.dumps(line)
    if OUT is not None:
        OUT.emit(text)
    else:
        print(text, flush=True)


def main():
    global OUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--envs", type=int, default=None, help="envs per GPU (default: the workload's)")
    ap.add_argument("--workload", default="C2", choices=["C2", "C4"])
    ap.add_argument("--actions", default="valid", choices=["valid", "any"],
                    help="BASELINE.md C2 series A (uniform random unrevealed cell, the bench line) or "
                         "series B (uniform random cell, includes no-op clicks)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="development: device-timed value and roofline only")
    ap.add_argument("--no-gae", action="store_true")
    ap.add_argument("--no-rollout", action="store_true")
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (a fixed, seeded sample of the envs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    set_workload(args.workload, args.envs)
    global VALID_ONLY
    VALID_ONLY = args.actions == "valid"

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    OUT = _QuietStdout()

    if args.impl == "reference":
        try:
            run_reference_arm(args, rank, world)
        finally:
            OUT.close()
        return

    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_cuda_arm(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        OUT.close()


if __name__ == "__main__":
    main()
