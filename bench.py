#!/usr/bin/env python
"""bench.py -- train rows/sec of the N x 128 least-squares fit (BASELINE.json `metric`).

One "step" = one complete fit of the resident rows through the C-ABI (b2_fit): four kernel launches --
    tc_shift_kernel     per-column shift from a 2048-row sample
    gram_tc_kernel      tcgen05 Gram over every row of this rank's shard (the roofline kernel)
    tc_finalize_kernel  reduce the per-CTA partials, fold into S, store S into every peer's exchange slot over NVLink (2-4 GPUs)
    solve kernel        waits for the peers' slots and sums them (2-4 GPUs), LDL^T, coefficients written to pinned host memory
At more than 4 GPUs the exchange is one ncclAllReduce of S between the finalize and the solve kernel instead: measured faster
there (profiles/r02_exchange_n8_diag.txt); `exchange.exchange_used` says which ran, B2_FORCE_P2P=1 / B2_NO_P2P=1 override.

Arms
    python bench.py [--gpus N --steps K --warmup W]          this repo (one process per GPU under torchrun)
                    [--dump-outputs DIR]                     + the last timed fit's coefficients and intercept as .npy
    python bench.py --impl reference [...]                   the reference's own CPU path: scikit-learn
                                                             LinearRegression.fit (stage_1_train_model.py:105-106)
                                                             on a bounded sample, all host threads, rank 0 only

Every N runs the SAME per-GPU shard (12.5 M x 128: BASELINE configs[2] over 8 GPUs), carries `parity` (the headline
fit against the exact fp64 kernel over the same full-size rows and the same exchange, S bit-identical across ranks) and
`exchange` (which exchange actually ran).  N = 1 adds `north_star` (100 M x 128 on one GPU), `config1_10Mx128`,
`companion_score`, `cpu_baseline`; N > 1 adds `strong_100M` and `score_shard`.  Keys follow the driver's contract; see
DESIGN.md "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D = 128
ROWS_CONFIG1 = 10_000_000      # BASELINE.json configs[1]
ROWS_PER_GPU = 12_500_000      # BASELINE.json configs[2]: 100 M rows over 8 GPUs -- the shard of every N (same-shard scaling)
NORTH_STAR_ROWS = 100_000_000  # BASELINE.json north_star: 100 M x 128 on one GPU
METRIC = "train rows/sec (N x 128 least-squares fit)"
UNIT = "rows/s"


# ---------------------------------------------------------------------------------------------------
def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """dense bf16 TFLOP/s (burst) of this pool's B200s, driver-written; fallback = the profiling recipe's figure"""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh).get("bf16_tflops", 1688.7))
    return 1688.7


def ncu_traffic_per_launch(workload_key: str):
    """dram bytes per launch of the Gram kernel from the committed ncu capture, if one matches."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh).get(workload_key)
    return None


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region, polled in-process through NVML every ~2 ms
    (the timed region of a 20-step run is ~20 ms -- too short for an `nvidia-smi -lms` subprocess to start).
    Falls back to the B200_PROFILING.md nvidia-smi recipe when pynvml is unavailable."""
    _REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
                ("hw_thermal_slowdown", 0x40), ("hw_power_brake_slowdown", 0x80))

    def __init__(self, device: int):
        self.device, self.samples, self.stop_flag, self.thread, self.h = device, [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            # torchrun may remap devices through CUDA_VISIBLE_DEVICES; NVML indexes physical devices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[device]) if vis and vis.split(",")[device].isdigit() else device
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                     nv.nvmlDeviceGetCurrentClocksEventReasons(self.h),
                                     nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0,
                                     nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_MEM)))
            except Exception:
                break
            time.sleep(0.002)

    def start(self):
        if self.nv is None:
            return
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.nv is None:
            return self._smi_once()
        self.stop_flag = True
        self.thread.join(timeout=2)
        if not self.samples:
            return self._smi_once()
        sm = sorted(s[0] for s in self.samples)
        mask = 0
        for s in self.samples:
            mask |= int(s[1])
        reasons = [name for name, bit in self._REASONS if mask & bit]
        try:
            mx = self.nv.nvmlDeviceGetMaxClockInfo(self.h, self.nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        mem = sorted(s[3] for s in self.samples)
        try:
            mem_mx = self.nv.nvmlDeviceGetMaxClockInfo(self.h, self.nv.NVML_CLOCK_MEM)
        except Exception:
            mem_mx = None
        # the HBM clock too: the Gram kernel's fraction of the (fixed) measured peak varies 0.8-0.97 box to box at equal SM clocks
        return {"sm_mhz": float(sm[len(sm) // 2]), "sm_max_mhz": float(mx) if mx else None, "samples": len(sm),
                "power_w_max": max(s[2] for s in self.samples), "reasons": reasons, "how": "NVML poll, 2 ms",
                "mem_mhz": float(mem[len(mem) // 2]), "mem_max_mhz": float(mem_mx) if mem_mx else None}

    def _smi_once(self) -> dict:
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                  str(self.device)], capture_output=True, text=True, timeout=10).stdout.strip()
            f = [x.strip() for x in out.split(",")]
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            return {"sm_mhz": float(f[0]), "sm_max_mhz": float(f[1]), "samples": 1, "power_w_max": float(f[2]),
                    "reasons": [n for n, v in zip(names, f[3:7]) if v.lower().startswith("active")],
                    "how": "nvidia-smi, one sample right after the timed region"}
        except Exception as exc:  # pragma: no cover
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"unavailable: {exc}"]}


# ---------------------------------------------------------------------------------------------------
def sklearn_fit_rows_per_s(rows: int, repeats: int = 1, seed: int = 1234):
    """The reference's fit call on `rows` x 128 fp32 rows drawn from the reference DGP; all host threads."""
    from sklearn.linear_model import LinearRegression
    from oracle import ols_oracle as orc
    X, y = orc.generate_dataset(rows, D, seed=seed, dtype=np.float32)
    best = float("inf")
    coef = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        reg = LinearRegression(fit_intercept=True).fit(X, y)
        best = min(best, time.perf_counter() - t0)
        coef = reg.coef_
    return rows / best, best, coef


def host_threads() -> int:
    try:
        from threadpoolctl import threadpool_info
        n = [p.get("num_threads", 0) for p in threadpool_info() if p.get("user_api") == "blas"]
        if n:
            return int(max(n))
    except Exception:
        pass
    return os.cpu_count() or 1


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import sklearn  # noqa: F401  (the reference's dependency; pinned 0.24.0 upstream, 1.9.0 in this image)
    try:   # torchrun exports OMP_NUM_THREADS=1: give the CPU arm every host thread BLAS will take
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count())
    except Exception:
        pass
    t_cal = sklearn_fit_rows_per_s(32_768)[1]
    budget = 150.0 / max(args.steps + args.warmup, 1)
    rows = int(min(1_000_000, max(32_768, 32_768 * budget / max(t_cal, 1e-3) * 0.5)))
    rows = (rows // 32_768) * 32_768
    from sklearn.linear_model import LinearRegression
    from oracle import ols_oracle as orc
    X, y = orc.generate_dataset(rows, D, seed=1234, dtype=np.float32)
    for _ in range(args.warmup):
        LinearRegression(fit_intercept=True).fit(X, y)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        LinearRegression(fit_intercept=True).fit(X, y)
    dt = time.perf_counter() - t0
    value = rows * args.steps / dt
    cores = host_threads()
    sample = f"{rows} x {D} fp32 rows of the same synthetic distribution per step (bounded sample of the workload)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus, "f32"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "what": "sklearn.linear_model.LinearRegression(fit_intercept=True).fit "
                                 "(stage_1_train_model.py:105-106; LAPACK gelsd), called as the oracle port does"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def workload_config(n_gpus: int, x_kind: str, rows: int = 0) -> dict:
    rows = rows or ROWS_PER_GPU
    return {"workload": (f"{rows * n_gpus} rows x {D} features ({rows} per GPU, row-sharded), X {x_kind} + y fp32 "
                         f"resident in HBM; the per-GPU shard of BASELINE.json configs[2] (100 M x 128 over 8 GPUs) at "
                         f"every N, so the driver's efficiency is same-shard; configs[1] (10 M x 128) is the "
                         f"`config1_10Mx128` object of the N = 1 line"),
            "rows_per_gpu": rows, "features": D, "x_storage": x_kind,
            "parallelism": f"row-shard x{n_gpus}, one exchange of the (D+2)^2 fp64 statistic per fit",
            "l2": f"inputs larger than L2 ({rows * (D * (4 if x_kind == 'f32' else 2) + 4) / 1e9:.2f} GB per pass vs 126 MB)"}


def max_over_ranks(dist, value: float) -> float:
    if dist is None:
        return value
    import torch
    t = torch.tensor([value], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def gather_ranks(dist, value: float):
    """`value` of every rank (gloo all-gather), rank order; None on one GPU."""
    if dist is None:
        return None
    import torch
    out = [torch.zeros(1, dtype=torch.float64) for _ in range(dist.get_world_size())]
    dist.all_gather(out, torch.tensor([value], dtype=torch.float64))
    return [round(float(t.item()), 5) for t in out]


def time_fits(ctx, dist, X, y, steps: int, warmup: int, barrier):
    """`steps` complete fits (b2_fit: Gram + exchange + solve, coefficients on the host), CUDA-event timed, max over
    ranks.  Returns (ms_total, gram_kernel_ms_avg, launches, last (coef, intercept))."""
    for _ in range(warmup):
        sol = ctx.fit(X, y)
    ctx.last_kernel_ms()
    l0 = ctx.launch_count()
    barrier()
    host_ms = []
    ctx.timer_start()
    for _ in range(steps):
        t0 = time.perf_counter()
        sol = ctx.fit(X, y)
        host_ms.append(1e3 * (time.perf_counter() - t0))
    ms = ctx.timer_stop()
    barrier()
    kms, kl = ctx.last_kernel_ms()
    time_fits.last_host_ms = host_ms
    return max_over_ranks(dist, ms), kms / max(kl, 1), ctx.launch_count() - l0, sol


def exact_check(ctx, b2, X, y, d, sol, dist, tag: str) -> dict:
    """Oracle check of a full-size fit: the same rows through the exact fp64 CUDA-core kernel (KERNEL_SIMT -- pinned to the
    numpy oracle at 1e-12 by tests/ and, in this run, by `oracle_pin`), the same exchange, the same solve."""
    coef, b0 = sol
    S_head = ctx.gram_export()
    ctx.set_kernel(b2.KERNEL_SIMT)
    ctx.sync()
    t0 = time.perf_counter()
    ctx.gram_reset(d); ctx.gram_accumulate(X, y); ctx.gram_allreduce()
    c_ex, b_ex = ctx.solve()
    secs = time.perf_counter() - t0
    S_ex = ctx.gram_export()
    ctx.set_kernel(b2.KERNEL_TCGEN05)
    out = {"what": f"{tag}: headline fit vs the exact fp64 kernel over the SAME full-size rows + the same exchange",
           "coef_linf": float(np.max(np.abs(coef - c_ex))), "intercept_abs_err": float(abs(b0 - b_ex)),
           "statistic_rel_err": float(np.max(np.abs(S_head - S_ex)) / np.max(np.abs(S_ex))),
           "rows_in_statistic": float(S_head[d, d]), "exact_kernel_seconds": secs, "tolerance": 1e-4}
    if dist is not None:
        import hashlib
        hs = [None] * dist.get_world_size()
        dist.all_gather_object(hs, hashlib.sha256(S_head.tobytes() + coef.tobytes()).hexdigest())
        out["bit_identical_across_ranks"] = bool(all(h == hs[0] for h in hs))
    return out


def dump_outputs(out_dir: str, coef, b0: float) -> None:
    """What the timed fit hands its caller: the coefficients and the intercept of the last step."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "coef.npy"), np.asarray(coef, dtype=np.float64))
    np.save(os.path.join(out_dir, "intercept.npy"), np.array([b0], dtype=np.float64))


# ---------------------------------------------------------------------------------------------------
def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--x-dtype", default="f32", choices=["f32", "bf16"])
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU (default: 12.5 M, the configs[2] shard)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip north_star / strong_100M / config1 variants / companion (profiling runs)")
    ap.add_argument("--no-variants", action="store_true", help="alias of --no-extras")
    ap.add_argument("--precision", default="split", choices=["split", "bf16"],
                    help="tensor-core operand precision: bf16 hi+lo split (default) or a single bf16 operand")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed fit's result to DIR/coef.npy and DIR/intercept.npy (float64); the "
                         "inputs are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    extras = not (args.no_extras or args.no_variants)

    if args.impl == "reference":
        run_reference(args)
        return

    import bodywork_mlops_demo_b200 as b2

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N > 1 with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N")
        args.gpus = world

    dist = None
    if world > 1:
        import torch  # noqa: F401
        import torch.distributed as dist  # rendezvous / barrier / max-over-ranks only (gloo, CPU tensors)
        dist.init_process_group("gloo", init_method="env://", rank=rank, world_size=world)

    ctx = b2.Context(local_rank)
    exchange_note = None
    if world > 1:
        uid = [b2.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        # NCCL may print its version banner on stdout; stdout carries exactly one JSON line, so park fd 1 on stderr
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            ctx.comm_init(world, rank, uid[0])
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
        # which exchange: measured on 8 GPUs, alternating runs on one box (profiles/r02_exchange_n8_diag.txt): NCCL 1.18-1.20 ms
        # per fit, the peer-memory exchange 1.39-1.51 ms (its system-scope fences do not scale with the number of peers);
        # at 2 and 4 GPUs the two are within 1-2 %.  So: peer-memory exchange up to 4 ranks, NCCL beyond;
        # B2_FORCE_P2P=1 / B2_NO_P2P=1 override.
        want_p2p = os.environ.get("B2_NO_P2P") != "1" and world <= 8 and (world <= 4 or os.environ.get("B2_FORCE_P2P") == "1")
        if want_p2p:
            # one-shot peer-memory exchange of S (NVLink stores + flags) fused into the Gram / solve kernels
            try:
                mine = ctx.comm_p2p_export()
            except Exception as exc:   # e.g. CUDA IPC unavailable in this container
                exchange_note = f"rank {rank}: peer-memory export failed ({exc})"
                mine = None
            handles = [None] * world
            dist.all_gather_object(handles, mine)          # every rank takes part in both collectives
            ok = all(h is not None for h in handles)
            if ok:
                try:
                    ctx.comm_p2p_attach(world, rank, handles)
                except Exception as exc:
                    exchange_note = f"rank {rank}: attaching peer buffers failed ({exc})"
                    ok = False
            oks = [None] * world
            dist.all_gather_object(oks, ok)                # also the barrier between attach and the first exchange
            if not all(oks):
                ctx.comm_p2p_detach()
                exchange_note = (exchange_note or "a peer could not attach") + "; NCCL all-reduce used"
        else:
            exchange_note = ("B2_NO_P2P=1: NCCL all-reduce" if os.environ.get("B2_NO_P2P") == "1" else
                             f"{world} ranks: NCCL all-reduce (measured faster than the peer-memory exchange beyond 4 ranks; "
                             f"B2_FORCE_P2P=1 selects the latter)")
        if exchange_note:
            print(f"[bench] {exchange_note}", file=sys.stderr)

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()
            # gloo releases the ranks milliseconds apart, and the first exchange of a timed loop absorbs that skew (a
            # 5-fit loop showed +70 % at N = 4); an NCCL all-reduce + stream sync aligns them to microseconds
            ctx.comm_barrier()

    rows = args.rows or ROWS_PER_GPU
    kind = args.x_dtype
    X, y = ctx.synth(rows, D, seed=1234, row_offset=rank * rows, kind=kind)
    ctx.set_kernel(b2.KERNEL_TCGEN05)
    ctx.set_precision(b2.PRECISION_BF16 if args.precision == "bf16" else b2.PRECISION_SPLIT)
    ctx.sync()
    peak, peak_src = measured_peaks()
    bytes_per_row = D * (4 if kind == "f32" else 2) + 4
    mma_per_row = 2.0 * 128 * 144 * (2 if args.precision == "split" else 1)

    # ---- headline: `steps` complete fits of the resident shard --------------------------------------------------
    for _ in range(args.warmup):
        coef, b0 = ctx.fit(X, y)
    ctx.last_kernel_ms()
    launches0 = ctx.launch_count()
    fused0 = ctx.stats()["fused_fits"]
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    ctx.timer_start()
    t_host0 = time.perf_counter()
    for _ in range(args.steps):
        coef, b0 = ctx.fit(X, y)
    ms = ctx.timer_stop()
    t_host = time.perf_counter() - t_host0
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:      # every rank solves the same all-reduced statistic
        dump_outputs(args.dump_outputs, coef, b0)
    kernel_ms, kernel_launches = ctx.last_kernel_ms()
    launches = ctx.launch_count() - launches0
    fused_fits = ctx.stats()["fused_fits"] - fused0
    step_ms_by_rank = gather_ranks(dist, ms / args.steps)
    kernel_ms_by_rank = gather_ranks(dist, kernel_ms / max(kernel_launches, 1))
    ms = max_over_ranks(dist, ms)

    total_rows = rows * world
    value = total_rows * args.steps / (ms * 1e-3)
    gram_ms = kernel_ms / max(kernel_launches, 1)
    achieved = rows * bytes_per_row / (gram_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "gram_tc_kernel",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                "mma_tflops_issued": rows * mma_per_row / gram_ms / 1e9,
                "algorithmic_bytes_per_row": bytes_per_row, "rows_per_launch": rows,
                "kernel_ms_avg": gram_ms, "kernel_share_of_step": gram_ms / (ms / args.steps),
                "step_tail_us": 1e3 * (ms / args.steps - gram_ms),
                "whole_fit_frac_of_hbm_peak": rows * bytes_per_row / (ms / args.steps * 1e-3) / 1e9 / peak,
                "traffic": ncu_traffic_per_launch(f"{kind}_{rows}x{D}")}
    try:       # this box's own copy bandwidth next to the pool's figure: the fraction above varies 0.8-0.97 box to box
        box = ctx.copy_bandwidth_gbs()
        roofline["copy_gbs_this_gpu"] = box
        roofline["frac_of_this_gpu_copy"] = achieved / box
    except Exception:  # noqa: BLE001 - a diagnostic, never fatal
        pass
    if kernel_ms_by_rank is not None:      # the step waits for the slowest rank: its kernel, not rank 0's, sets the tail
        roofline["kernel_ms_by_rank"] = kernel_ms_by_rank
        roofline["step_ms_by_rank"] = step_ms_by_rank
        roofline["step_tail_us_vs_slowest_kernel"] = 1e3 * (ms / args.steps - max(kernel_ms_by_rank))
    info = ctx.comm_info()
    exchange = {"exchange_used": info["exchange"], "n_ranks": info["n_ranks"], "note": exchange_note,
                "fused_fits": fused_fits, "of_steps": args.steps,
                "launches_per_step": launches / max(args.steps, 1)}

    # ---- parity of the HEADLINE fit at this N: exact kernel over the same rows + the same exchange ------------------
    parity = exact_check(ctx, b2, X, y, D, (coef, b0), dist, f"{total_rows} x {D}")
    parity["rows_expected"] = float(total_rows)
    parity["row_count_exact"] = bool(parity["rows_in_statistic"] == float(total_rows))

    # ---- sharded scoring: b2_score per shard + b2_score_allreduce, checked against the host-side combination ----------
    score_shard = None
    if world > 1:
        ctx.set_kernel(b2.KERNEL_AUTO)
        _yh, st_local = ctx.score(X, coef, float(b0), y=y, want_yhat=False)
        st_all = ctx.score_allreduce(st_local.copy())
        parts = [None] * world
        dist.all_gather_object(parts, st_local.tolist())
        want = b2.sharding.combine_score_stats(np.array(parts))
        score_shard = {"what": "b2_score on every shard + b2_score_allreduce (8 sums + 2 maxima over NCCL) vs the "
                               "combination of the per-rank statistics gathered over gloo",
                       "rel_err": float(np.max(np.abs(st_all - want) / np.maximum(np.abs(want), 1e-300))),
                       "rows": float(st_all[5]),
                       "r_squared": float(1.0 - st_all[1] / max(st_all[3] - st_all[2] ** 2 / max(st_all[5], 1.0), 1e-300))}
        ctx.set_kernel(b2.KERNEL_TCGEN05)

    # ---- the north-star point (N = 1): 100 M x 128 fp32 on ONE GPU; strong scaling of the same 100 M rows (N > 1) ------
    north_star = None
    strong = None
    if extras and kind == "f32":
        ns_rows = NORTH_STAR_ROWS // world
        if world == 1 or ns_rows != rows:
            Xn, yn = ctx.synth(ns_rows, D, seed=1234, row_offset=rank * ns_rows, kind="f32")
            ns_sampler = ClockSampler(local_rank)
            if rank == 0:
                ns_sampler.start()
            ns_ms, ns_kms, _l, ns_sol = time_fits(ctx, dist, Xn, yn, 5, 3, barrier)
            ns_clocks = ns_sampler.stop() if rank == 0 else None
            chk = exact_check(ctx, b2, Xn, yn, D, ns_sol, dist, f"{ns_rows * world} x {D}")
            rec = {"rows_total": ns_rows * world, "rows_per_gpu": ns_rows, "ms_per_fit": ns_ms / 5,
                   "fit_rows_per_s": ns_rows * world / (ns_ms / 5) * 1e3, "gram_kernel_ms": ns_kms,
                   "gram_kernel_frac_of_hbm_peak": ns_rows * 516 / ns_kms / 1e6 / peak,
                   "whole_fit_frac_of_hbm_peak": ns_rows * 516 / (ns_ms / 5) / 1e6 / peak,
                   "coef_linf_vs_exact": chk["coef_linf"], "intercept_abs_err_vs_exact": chk["intercept_abs_err"],
                   "statistic_rel_err": chk["statistic_rel_err"], "rows_in_statistic": chk["rows_in_statistic"],
                   "exact_kernel_seconds": chk["exact_kernel_seconds"],
                   "bit_identical_across_ranks": chk.get("bit_identical_across_ranks"),
                   "coef_head": [float(c) for c in ns_sol[0][:3]], "intercept": float(ns_sol[1]),
                   "per_fit_host_ms": [round(v, 3) for v in time_fits.last_host_ms], "clocks": ns_clocks}
            Xn.free(); yn.free()
        else:
            rec = {"rows_total": total_rows, "rows_per_gpu": rows, "ms_per_fit": ms / args.steps,
                   "fit_rows_per_s": value, "note": "identical to the headline line (100 M rows over 8 GPUs)",
                   "coef_linf_vs_exact": parity["coef_linf"]}
        if world == 1:
            rec["what"] = ("BASELINE.json north_star: >= 70 % of the HBM roofline on the Gram kernel at N = 100 M, "
                           "D = 128 on 1 B200, coefficient error < 1e-4")
            north_star = rec
        else:
            rec["what"] = (f"SURVEY 8(d) config 3: the SAME 100 M x 128 rows strong-scaled over {world} GPUs "
                           f"(1 GPU: the `north_star` object of the N = 1 line)")
            strong = rec

    # ---- e2e: the public estimator API with DEFAULT arguments on HOST rows; H2D inside the timed region -------------
    e2e = None
    if not args.no_e2e:
        Xp = ctx.pinned((rows, D), np.float32 if kind == "f32" else np.uint16)
        yp = ctx.pinned((rows,), np.float32)
        b2.native._check(b2.native.load().b2_copy_d2h(ctx._h, Xp.ptr, X.ptr, X.nbytes), "d2h X")
        b2.native._check(b2.native.load().b2_copy_d2h(ctx._h, yp.ptr, y.ptr, y.nbytes), "d2h y")
        est = b2.B200LinearRegression(ctx=ctx)
        ctx.set_kernel(b2.KERNEL_AUTO)
        e2e_steps = max(2, min(args.steps, 4))
        est.fit(Xp.array, yp.array)                    # warm-up (allocates the staging ring)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            est.fit(Xp.array, yp.array)                # default arguments: coefficients AND singular_ / rank_
        dt = time.perf_counter() - t0
        barrier()
        dt = max_over_ranks(dist, dt)
        e2e = {"value": total_rows * e2e_steps / dt, "unit": UNIT, "steps": e2e_steps,
               "h2d_bytes_per_step": int(rows * bytes_per_row), "d2h_bytes_per_step": int((2 * D + 8) * 8 * 2),
               "api": "B200LinearRegression().fit(X_host_pinned, y_host_pinned), default arguments (coef_, intercept_, "
                      "singular_, rank_) -> b2_fit(B2_MEM_HOST) + b2_solve_eigvals",
               "coef_linf_vs_resident": float(np.max(np.abs(est.coef_ - coef))), "rank_": int(est.rank_)}
        if world == 1 and extras:
            # the same call on ordinary (pageable) numpy rows -- what train_model hands over -- and train_model itself
            m = min(rows, 2_000_000)
            Xn, yn = np.array(Xp.array[:m]), np.array(yp.array[:m])
            if kind == "f32":
                est.fit(Xn, yn)
                t0 = time.perf_counter()
                for _ in range(3):
                    est.fit(Xn, yn)
                e2e["pageable_rows_per_s"] = m * 3 / (time.perf_counter() - t0)
                e2e["pageable_sample"] = f"{m} x {D} fp32 rows in pageable host memory, default fit()"
                import pandas as pd
                from bodywork_mlops_demo_b200 import stage_1_train_model as s1
                # float64 host rows, the scikit-learn habit (converted by b2_upload_columns on the way up)
                X64, y64 = Xn.astype(np.float64), yn.astype(np.float64)
                est.fit(X64, y64)
                f64_ms = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    est.fit(X64, y64)
                    f64_ms.append(1e3 * (time.perf_counter() - t0))
                e2e["float64_rows_per_s"] = m / (min(f64_ms) * 1e-3)
                e2e["float64_fit_ms"] = [round(v, 1) for v in f64_ms]
                e2e["float64_sample"] = f"{m} x {D} float64 rows in pageable host memory, default fit()"
                mt = 500_000
                # the reference's input: a float64 DataFrame (what pd.read_csv yields), through the stage's own train_model
                df = pd.DataFrame({"date": "2021-01-01", "y": y64[:mt], **{f"X{j}": X64[:mt, j] for j in range(D)}})
                s1.train_model(df)
                t0 = time.perf_counter()
                model, metrics = s1.train_model(df)
                e2e["train_model_rows_per_s"] = mt / (time.perf_counter() - t0)
                e2e["train_model_sample"] = (f"stage_1 train_model(float64 DataFrame {mt} x {D}): columns -> b2_upload_columns, "
                                             f"split mask + masked fit + hold-out scoring + sklearn artefact; "
                                             f"r_squared {float(metrics['r_squared'][0]):.4f}")
                del df, X64, y64
        Xp.free(); yp.free()
        ctx.set_kernel(b2.KERNEL_TCGEN05)

    # ---- BASELINE configs[1]: 10 M x 128 on one GPU, every storage x operand combination ---------------------------
    config1 = None
    if world == 1 and extras:
        config1 = {"what": "BASELINE.json configs[1]: 10 M x 128 rows resident on one GPU; complete fits (b2_fit); bf16-stored "
                           "rows run gram_b16_kernel; coef_linf_vs_exact: against the exact fp64 kernel over the same stored rows",
                   "rows": ROWS_CONFIG1}
        exact_c1 = {}
        for vk, vprec in (("f32", "split"), ("f32", "bf16"), ("bf16", "split"), ("bf16", "bf16")):
            Xv, yv = ctx.synth(ROWS_CONFIG1, D, seed=1234, kind=vk)
            ctx.set_precision(b2.PRECISION_BF16 if vprec == "bf16" else b2.PRECISION_SPLIT)
            vms, vk_ms, _l, vsol = time_fits(ctx, None, Xv, yv, 10, 3, barrier)
            bpr = D * (4 if vk == "f32" else 2) + 4
            mma = 2.0 * 128 * 144 * (1 if vprec == "bf16" else 2)
            config1[f"x_{vk}_operands_{'bf16x1' if vprec == 'bf16' else 'bf16x2'}"] = {
                "fit_rows_per_s": ROWS_CONFIG1 / (vms / 10) * 1e3, "ms_per_fit": vms / 10, "gram_kernel_ms": vk_ms,
                "frac_of_hbm_peak": ROWS_CONFIG1 * bpr / vk_ms / 1e6 / peak,
                "mma_tflops_issued": ROWS_CONFIG1 * mma / vk_ms / 1e9,
                "frac_of_bf16_tensor_peak": ROWS_CONFIG1 * mma / vk_ms / 1e9 / measured_tensor_peak(),
                "coef_head": [float(c) for c in vsol[0][:2]]}
            if vk not in exact_c1:          # the exact fp64 kernel over the same stored rows, once per storage type
                ctx.set_kernel(b2.KERNEL_SIMT)
                ctx.gram_reset(D); ctx.gram_accumulate(Xv, yv)
                exact_c1[vk] = ctx.solve()[0]
                ctx.set_kernel(b2.KERNEL_TCGEN05)
            config1[f"x_{vk}_operands_{'bf16x1' if vprec == 'bf16' else 'bf16x2'}"]["coef_linf_vs_exact"] = \
                float(np.max(np.abs(vsol[0] - exact_c1[vk])))
            Xv.free(); yv.free()
        ctx.set_precision(b2.PRECISION_BF16 if args.precision == "bf16" else b2.PRECISION_SPLIT)

    # ---- the estimator's DEFAULT fit on the resident shard: coefficients AND singular_ / rank_ (eigenvalue kernel) ----
    default_fit = None
    if world == 1 and extras:
        est_d = b2.B200LinearRegression(ctx=ctx)
        for _ in range(2):
            est_d.fit(X, y)
        ctx.sync(); ctx.timer_start()
        for _ in range(10):
            est_d.fit(X, y)
        dms = ctx.timer_stop() / 10
        default_fit = {"what": "B200LinearRegression().fit(X_dev, y_dev), default arguments, resident rows: b2_fit + "
                               "b2_solve_eigvals (singular_, rank_ of the sklearn artefact)",
                       "ms_per_fit": dms, "rows_per_s": rows / dms * 1e3, "spectrum_ms": dms - ms / args.steps,
                       "rank_": int(est_d.rank_), "singular_head": [float(v) for v in est_d.singular_[:2]]}

    # ---- companion kernel: hold-out scoring + metrics over the same resident rows (stage_1...:107, 79-90) ----------
    companion = None
    if world == 1 and extras:
        ctx.set_kernel(b2.KERNEL_AUTO)
        for _ in range(3):
            ctx.score(X, coef, float(b0), y=y, want_yhat=False)
        ctx.sync(); ctx.timer_start()
        for _ in range(10):
            _yh, sstats = ctx.score(X, coef, float(b0), y=y, want_yhat=False)
        sms = ctx.timer_stop() / 10
        companion = {"what": "b2_score: X.coef + intercept fused with the ten metric reductions, resident rows, no yhat write",
                     "ms": sms, "rows_per_s": rows / sms * 1e3, "bytes_per_row": bytes_per_row,
                     "frac_of_hbm_peak": rows * bytes_per_row / sms / 1e6 / peak,
                     "note": "timed with CUDA events around 10 calls; includes the 80-byte D2H of the statistics per call",
                     "r_squared": float(1.0 - sstats[1] / max(sstats[3] - sstats[2] ** 2 / max(sstats[5], 1.0), 1e-300))}
        ctx.set_kernel(b2.KERNEL_TCGEN05)

    # ---- CPU baseline + oracle pin: numpy / sklearn on the host cores, bounded samples, rank 0 ------------------------
    cpu = None
    oracle_pin = None
    if rank == 0 and not args.no_cpu_baseline:
        try:   # torchrun exports OMP_NUM_THREADS=1
            from threadpoolctl import threadpool_limits
            threadpool_limits(limits=os.cpu_count())
        except Exception:
            pass
        from oracle import ols_oracle as orc
        from sklearn.linear_model import LinearRegression
        # (1) the exact kernel IS the numpy oracle: statistic of the first rows of this rank's shard, both ways
        m = 400_000
        lib = b2.native.load()
        es = 4 if kind == "f32" else 2
        Xh = np.empty((m, D), dtype=np.float32 if kind == "f32" else np.uint16)
        yh = np.empty(m, dtype=np.float32)
        b2.native._check(lib.b2_copy_d2h(ctx._h, Xh.ctypes.data, X.ptr, m * D * es), "d2h X head")
        b2.native._check(lib.b2_copy_d2h(ctx._h, yh.ctypes.data, y.ptr, m * 4), "d2h y head")
        Xf = Xh.astype(np.float64) if kind == "f32" else b2.native.from_bf16_bits(Xh).astype(np.float64)
        S_np = orc.gram_stats(Xf, yh.astype(np.float64))
        # a second context (no communicator): the statistic / fit of the slice alone, exact kernel and tensor-core kernel
        c2 = b2.Context(local_rank)
        X2, y2 = c2.to_device(Xh, kind), c2.to_device(yh)
        c2.set_kernel(b2.KERNEL_SIMT)
        c2.gram_reset(D); c2.gram_accumulate(X2, y2)
        S_dev = c2.gram_export()
        c2.set_kernel(b2.KERNEL_TCGEN05)
        c_tc, b_tc = c2.fit(X2, y2)
        c2.close()
        reg = LinearRegression().fit(Xf[:200_000], yh[:200_000].astype(np.float64))
        ref = orc.fit_from_stats(S_np)
        oracle_pin = {"rows": m,
                      "exact_kernel_vs_numpy_oracle_statistic_rel": float(np.max(np.abs(S_dev - S_np)) / np.max(np.abs(S_np))),
                      "tensor_core_fit_vs_numpy_oracle_coef_linf": float(np.max(np.abs(c_tc - ref["coef"]))),
                      "tensor_core_fit_vs_numpy_oracle_intercept": float(abs(b_tc - ref["intercept"])),
                      "oracle_vs_sklearn_fp64_coef_linf_200k": float(np.max(np.abs(
                          orc.fit_from_stats(orc.gram_stats(Xf[:200_000], yh[:200_000].astype(np.float64)))["coef"] - reg.coef_))),
                      "tolerance": 1e-4}
        # (2) the reference's fit call, timed on the host cores
        if world == 1:
            sample_rows = 1_000_000
            v, secs, _ = sklearn_fit_rows_per_s(sample_rows)
            cpu = {"value": v, "unit": UNIT, "cores": host_threads(), "kind": "port", "seconds": secs,
                   "sample": f"{sample_rows} x {D} fp32 rows, one LinearRegression(fit_intercept=True).fit "
                             f"(stage_1_train_model.py:105-106), all BLAS threads"}
    if dist is not None:
        dist.barrier()

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": ("bf16x2 (hi+lo)" if args.precision == "split" else "bf16x1") + " MMA operands, f32 accumulate, f64 fold+solve",
            "data": "synthetic (device Philox, reference DGP: X~U(0,100), y=1+0.5*sum(X)+10*eps)",
            "config": workload_config(world, kind, rows), "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "oracle_pin": oracle_pin, "exchange": exchange,
            "score_shard": score_shard, "north_star": north_star, "strong_100M": strong, "config1_10Mx128": config1,
            "companion_score": companion, "default_fit_resident": default_fit,
            "host_wall_ms_per_step": 1e3 * t_host / args.steps,
            "coef_head": [float(c) for c in coef[:3]], "intercept": float(b0),
        }
        print(json.dumps(out))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
