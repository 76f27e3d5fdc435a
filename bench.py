#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native faer hot path.

N = 1 (BASELINE.json configs[1], the configuration the metric is quoted on): f64 Cholesky LLT, n = 16384, synthetic SPD
input A = G G^T + n I (G ~ N(0,1), the reference's bench generator, faer/examples/bench.rs:1513-1515), column-major,
resident in HBM when the timed region starts. One "step" = restore the input (device copy of the 2.1 GB matrix; faer's own
bench also times `copy_from_triangular_lower`, bench.rs:1531-1540) + one in-place factorisation through the C ABI
`libfaer_v0_23_llt_factor_in_place_f64`.
  value  = n^3/3 flop per factorisation (SURVEY.md §8d) / device time                          [TFLOP/s]
  e2e    = same metric through the same C-ABI call with HOST (pinned) buffers: H2D + factor + D2H inside the timed region
  configs2_lu_n32768 (mandatory block of the N = 1 line) = the 1-GPU point of the curve below: same matrix, same code.

N > 1 (torchrun, one rank per GPU; BASELINE.json configs[2]): f64 partial-pivoting LU of ONE n = 32768 Gaussian matrix by
all N GPUs — 1-D block-column-cyclic layout, NCCL broadcast of each factored panel + its transpositions with look-ahead
(csrc/dist.cu). STRONG scaling: the matrix (generated column chunk by column chunk from fixed seeds, so every N sees the
same bits) and the flop count 2 n^3 / 3 do not depend on N; value = 2 n^3 / 3 / (max-over-ranks device time). The line
carries a SHA-1 of `perm_fwd` (`config.perm_sha1`) — equal on every N and in the N = 1 block iff the pivots are identical —
and `p1_check`: rank 0 factors the whole matrix on its own GPU after the timed region and compares permutation (exact) and
factors with the distributed result. The previous round's workload (weak-scaled LLT) is kept in `also.llt_weak`.

--impl reference: times the CPU restatement of the reference's algorithm (oracle/, OpenMP over the host cores; faer itself
needs a Rust toolchain that this image does not have) — LLT at the SAME n = 16384 at N = 1, a bounded sample of the LU at
N > 1 (the port needs ~80 s for one n = 32768 factorisation).

--dump-outputs DIR (N = 1 GPU arm): after the timed steps, writes the Cholesky factor the last timed step left in A as
float64 .npy files, so that two builds can be compared output for output on the same seeded input:
  llt_factor_diagonal.npy  the n diagonal entries of L
  llt_factor_columns.npy   n x k: L's columns at k sorted indices drawn by numpy's default_rng(0) (all columns when they fit),
                           entries above the diagonal (not part of the factor) set to 0; k * n * 8 <= 32 MiB
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

METRIC = "f64 GEMM & LU/LLT TFLOP/s at n=16384; % of B200 tensor-core peak"
UNIT = "TFLOP/s"
N_DEFAULT = 16384


LU_N = 32768  # BASELINE.json configs[2]


def llt_flops(n: int) -> float:
    return n ** 3 / 3.0


def lu_flops(n: int) -> float:
    return 2.0 * n ** 3 / 3.0


# ---------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append((time.time(), line.strip()))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for (ts, line) in self.rows:
            if ts < t0 or ts > t1 + 0.2:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples inside the timed region"], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU legs (oracle = test infrastructure; this is one of the two places allowed to execute it)
# ---------------------------------------------------------------------------------------------------
def cpu_llt_sample(target_seconds: float = 15.0, n_cap: int = 12288):
    """Time the CPU restatement of faer's LLT on all host cores on a bounded sample (same generator, smaller n)."""
    from oracle import oracle as orc
    orc.load()
    # The restatement keeps faer's 128-wide recursion, i.e. many small OpenMP regions: beyond ~32 threads the fork/join
    # cost dominated on the GPU box (first version: 0.0007 TFLOP/s with 128 threads vs 0.017 with 64), so the team is
    # capped. Since then the products run cache-blocked on packed panels and the triangular solves fork once per solve
    # (bitwise the same results; 5x faster on 8 cores here), but the cap has not been re-measured on the box.
    cores = max(1, min(os.cpu_count() or 1, 32))
    orc.set_num_threads(cores)
    rng = np.random.default_rng(0)

    def run(n):
        G = rng.standard_normal((n, n))
        A = np.asfortranarray(G @ G.T + n * np.eye(n))
        t = time.perf_counter()
        fail, _ = orc.llt(A)
        dt = time.perf_counter() - t
        assert fail == -1
        return dt

    run(512)  # thread start-up
    t_probe = run(2048)
    rate = llt_flops(2048) / t_probe
    n = int((target_seconds * rate * 3.0) ** (1.0 / 3.0)) // 256 * 256
    n = max(2048, min(n_cap, n))
    dt = run(n)
    return {"value": llt_flops(n) / dt / 1e12, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"oracle (C++/OpenMP restatement of faer's LLT, not faer itself: no Rust toolchain) LLT n={n}, "
                      f"same generator as the GPU workload, {dt:.2f} s"}, n, dt


def lapack_proxy(n: int):
    """scipy/OpenBLAS dpotrf on all cores at the full size — a PROXY for an optimised CPU library, not faer."""
    try:
        import scipy.linalg as sla
        rng = np.random.default_rng(0)
        G = rng.standard_normal((n, n))
        A = np.asfortranarray(G @ G.T + n * np.eye(n))
        t = time.perf_counter()
        sla.cholesky(A, lower=True, overwrite_a=True, check_finite=False)
        dt = time.perf_counter() - t
        return {"value": llt_flops(n) / dt / 1e12, "unit": UNIT, "what": f"scipy.linalg.cholesky (OpenBLAS) n={n}, {dt:.2f} s",
                "cores": os.cpu_count()}
    except Exception as e:  # pragma: no cover
        return {"value": None, "what": f"unavailable: {e}"}


def cpu_lu_sample_n(target_seconds: float, orc) -> int:
    rng = np.random.default_rng(5)
    A = np.asfortranarray(rng.standard_normal((2048, 2048)))
    t = time.perf_counter(); orc.lu(A); dt = time.perf_counter() - t
    rate = lu_flops(2048) / dt
    n = int((target_seconds * rate * 1.5) ** (1.0 / 3.0)) // 256 * 256
    return max(2048, min(16384, n))


def run_reference_arm(args):
    """--impl reference: the reference's algorithm on the host cores (oracle port; faer cannot be built here).
    N = 1: LLT at the GPU arm's own n (same_config) unless that would take longer than ~4 minutes in total, in which case a
    bounded sample is used and the line says so. N > 1: the GPU arm's workload is the LU of configs[2] at n = 32768 (one
    factorisation of which takes the port more than a minute): bounded sample of the same generator."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as orc
    orc.load()
    cores = max(1, min(os.cpu_count() or 1, 32))
    orc.set_num_threads(cores)
    lu_mode = args.gpus > 1
    rng = np.random.default_rng(1)
    if lu_mode:
        n_full = args.n or LU_N
        n = min(n_full, cpu_lu_sample_n(4.0, orc))
        flops = lu_flops(n)
        kind = "partial-pivoting LU"
    else:
        n_full = args.n or N_DEFAULT
        base, _, _ = cpu_llt_sample(target_seconds=4.0, n_cap=4096)
        est = llt_flops(n_full) / (base["value"] * 1e12)  # seconds per full-size step at the sampled rate
        n = n_full if est * (args.steps + 1) <= 240.0 else max(2048, int(n_full * (240.0 / (est * (args.steps + 1))) ** (1 / 3.0)) // 256 * 256)
        flops = llt_flops(n)
        kind = "Cholesky LLT"
    times = []
    for it in range(1 + args.steps):  # one warm-up is enough for a CPU loop; keeps the whole run within minutes
        if lu_mode:
            A = np.asfortranarray(rng.standard_normal((n, n)))
        else:
            G = rng.standard_normal((n, n))
            A = np.asfortranarray(G @ G.T + n * np.eye(n))
            del G
        t = time.perf_counter()
        if lu_mode:
            orc.lu(A)
        else:
            orc.llt(A)
        dt = time.perf_counter() - t
        if it >= 1:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = flops / (ms * 1e-3) / 1e12
    same = (n == n_full)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": 1, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if lu_mode else "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": (f"f64 {kind} n={n}" + ("" if same else f" (bounded CPU sample of the n={n_full} workload)") +
                                ", oracle port (C++/OpenMP restatement of faer's algorithm; faer itself needs Rust, absent here)"),
                   "n": n, "n_full": n_full, "same_config": same},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"oracle {kind} n={n} per step, {len(times)} steps after 1 warm-up"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
LU_CHUNK = 256  # columns generated per seed: the matrix does not depend on N or on the block width


def lu_local_input(torch, dev, n: int, nb: int, world: int, rank: int, lay):
    """This rank's block columns of the n x n Gaussian matrix of configs[2]; returned as the column-major n x local_cols
    view of a (local_cols, n) tensor. Column chunk c (256 columns) comes from torch's Philox generator seeded 777 + c."""
    assert nb % LU_CHUNK == 0 and n % LU_CHUNK == 0
    blocks = lay.local_blocks(n, nb, world, rank)
    ncols = lay.local_cols(n, nb, world, rank)
    out = torch.empty((ncols, n), dtype=torch.float64, device=dev)
    g = torch.Generator(device=dev)
    o = 0
    for b in blocks:
        c0, c1 = b * nb, min(n, (b + 1) * nb)
        for c in range(c0 // LU_CHUNK, c1 // LU_CHUNK):
            g.manual_seed(777 + c)
            out[o:o + LU_CHUNK].copy_(torch.randn((LU_CHUNK, n), generator=g, dtype=torch.float64, device=dev))
            o += LU_CHUNK
    return out.T


def perm_sha1(perm) -> str:
    import hashlib
    return hashlib.sha1(np.ascontiguousarray(perm, dtype="<i8").tobytes()).hexdigest()[:16]


def run_lu(torch, dist, lay, lib, dev, stream, world, rank, local_rank, n, nb, steps, warmup, sample_clocks=True):
    """Times `steps` distributed (or single-GPU, world == 1) LU factorisations of the configs[2] matrix. Returns a dict."""
    A0 = lu_local_input(torch, dev, n, nb, world, rank, lay)
    A = A0.clone(memory_format=torch.preserve_format)
    out = {}
    perm = pinv = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        nonlocal perm, pinv
        A.copy_(A0)
        perm, pinv, _ = lay.lu_in_place(A, n, nb=nb)

    for _ in range(warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank) if sample_clocks else None
    if sampler:
        sampler.start()
        time.sleep(0.25)
    l0 = lib.faer_b200_launch_count()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.time()
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    barrier()
    t1 = time.time()
    out["launches"] = int(lib.faer_b200_launch_count() - l0)
    ms = e0.elapsed_time(e1)
    if sampler:
        out["clocks"] = sampler.stop(t0, t1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out["ms_per_step"] = float(t.item()) / steps
    out["value"] = lu_flops(n) / (out["ms_per_step"] * 1e-3) / 1e12
    out["perm_sha1"] = perm_sha1(perm)
    # ---- probe on the timed data: (P A) x == L (U x), reduced over the ranks ----
    gcols = torch.as_tensor(lay.global_col_indices(n, nb, world, rank), device=dev)
    torch.manual_seed(99)
    x = torch.randn((n, 2), dtype=torch.float64, device=dev)
    rows = torch.arange(n, device=dev)
    zero = torch.zeros((), dtype=torch.float64, device=dev)
    ax = A0 @ x[gcols, :]
    ux = torch.where(rows[:, None] <= gcols[None, :], A, zero) @ x[gcols, :]
    amax = A0.abs().max().reshape(1); umax = ux.abs().max().reshape(1)
    if world > 1:
        dist.all_reduce(ax); dist.all_reduce(ux); dist.all_reduce(amax, op=dist.ReduceOp.MAX)
    Lloc = torch.where(rows[:, None] > gcols[None, :], A, zero)
    Lloc[gcols, torch.arange(gcols.numel(), device=dev)] = 1.0
    lux = Lloc @ ux[gcols, :]
    if world > 1:
        dist.all_reduce(lux)
    pax = ax[torch.as_tensor(perm, device=dev), :]
    out["probe_residual"] = float((pax - lux).abs().max()) / (float(amax.item()) * n)
    del Lloc
    out["_A0"], out["_A"], out["_perm"] = A0, A, perm
    return out


DUMP_COLUMN_BYTES = 32 << 20  # sampled columns of the factor written by --dump-outputs


def dump_llt_factor(torch, A, out_dir: str) -> None:
    """Writes the diagonal and a fixed, seeded sample of columns of the lower-triangular factor held in A (see --dump-outputs)."""
    n = A.shape[0]
    k = min(n, max(1, DUMP_COLUMN_BYTES // (8 * n)))
    cols = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
    idx = torch.as_tensor(cols, device=A.device)
    rows = torch.arange(n, device=A.device)
    L = torch.where(rows[:, None] >= idx[None, :], A[:, idx], torch.zeros((), dtype=A.dtype, device=A.device))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "llt_factor_diagonal.npy"), torch.diagonal(A).cpu().numpy())
    np.save(os.path.join(out_dir, "llt_factor_columns.npy"), L.cpu().numpy())


DIST_NB = 1024
LU_NB = 512   # block-column width of the LU runs (configs[2])


def weak_n(world: int, nb: int = DIST_NB) -> int:
    """Weak scaling: per-GPU flop (n^3 / 3 / N) held at the N=1 value => n ~ 16384 * N^(1/3), rounded to whole blocks."""
    if world == 1:
        return N_DEFAULT
    return int(round(N_DEFAULT * world ** (1.0 / 3.0) / nb)) * nb


def main_lu_strong(args, torch, dist, faer_b200, lay, lib, dev, stream, world, rank, local_rank):
    """N > 1: BASELINE.json configs[2] — one n = 32768 f64 partial-pivoting LU on all N GPUs, strong scaling."""
    import ctypes as C
    n = args.n or LU_N
    nb = args.nb if args.nb != DIST_NB else LU_NB
    r = run_lu(torch, dist, lay, lib, dev, stream, world, rank, local_rank, n, nb, args.steps, args.warmup)
    A0, A, perm = r.pop("_A0"), r.pop("_A"), r.pop("_perm")

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    # ---- roofline of the dominant kernel (the trailing-update GEMM), rank 0's launches, look-ahead overlap off ----
    A.copy_(A0)
    lib.faer_b200_profile_begin()
    lay.lu_in_place(A, n, nb=nb, lookahead=False)
    barrier()
    flops = C.c_double(0); ms = C.c_double(0); cnt = C.c_ulonglong(0)
    lib.faer_b200_profile_end(C.byref(flops), C.byref(ms), C.byref(cnt))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "profiles", "r01_f64_peaks.json")))
    except Exception:
        pass
    peak = peaks.get("dmma_tflops_sustained", 36.9)
    ach = flops.value / (ms.value * 1e-3) / 1e12 if ms.value > 0 else None
    roof = {"bound": "tensor", "kernel": "gemm_f64_ws_kernel / gemm_f64_kernel (DMMA.8x8x4; trailing updates A22 -= L21 U12 of this rank's "
                                          "block columns, k = nb)",
            "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": (ach / peak) if ach else None, "traffic": None,
            "launches_per_step": int(cnt.value), "ms_in_kernel_per_step": ms.value, "flops_in_kernel_per_step": flops.value,
            "peak_source": "measured on this pool: DMMA.8x8x4 issue-bound peak per GPU, profiles/r01_f64_peaks.json",
            "how": "CUDA events around every GEMM launch of rank 0 during one extra step after the timed region, look-ahead "
                   "overlap off; achieved = sum(algorithmic flop per launch) / sum(duration) on ONE GPU"}

    # ---- e2e: this rank's block columns start and end in pinned HOST memory, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        cols_, rows_ = A0.shape[1], A0.shape[0]
        hA0 = torch.empty((cols_, rows_), dtype=torch.float64, pin_memory=True)
        hA0.copy_(A0.T)
        hA = torch.empty((cols_, rows_), dtype=torch.float64, pin_memory=True)
        dA = torch.empty((cols_, rows_), dtype=torch.float64, device=dev)

        def e2e_call():
            dA.copy_(hA, non_blocking=True)
            lay.lu_in_place(dA.T, n, nb=nb)
            hA.copy_(dA, non_blocking=True)
            torch.cuda.synchronize()
        hA.copy_(hA0); e2e_call()
        ts = []
        for _ in range(max(2, min(args.steps, 3))):
            hA.copy_(hA0)
            barrier()
            t0 = time.perf_counter()
            e2e_call()
            ts.append(time.perf_counter() - t0)
        tt = torch.tensor([float(np.mean(ts))], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": lu_flops(n) / float(tt.item()) / 1e12, "unit": UNIT, "h2d_bytes_per_step": n * n * 8,
               "d2h_bytes_per_step": n * n * 8 + 2 * n * 8, "ms_per_step": 1e3 * float(tt.item()),
               "how": "faer_b200.dist.lu_in_place (faer_b200_dist_partial_piv_lu_factor_in_place_f64) on each rank's block columns; "
                      "pinned host -> device copy of the columns, factorisation, device -> host copy of the factors and the "
                      "permutations, wall clock, max over ranks"}
        del hA, hA0, dA

    # ---- P = 1 check on rank 0: the whole matrix on one GPU, same block width; permutation exact, factors compared ----
    p1 = None
    try:
        if rank == 0:
            F0 = lu_local_input(torch, dev, n, nb, 1, 0, lay)
            pf, _, _ = lay.lu_in_place(F0, n, nb=nb, lookahead=3)  # bit 1: ignore the communicator
            gcols = torch.as_tensor(lay.global_col_indices(n, nb, world, 0), device=dev)
            diff = float((F0[:, gcols] - A).abs().max())
            scale = float(F0[:, gcols].abs().max())
            p1 = {"perm_equal": bool(np.array_equal(pf, perm)), "perm_sha1_p1": perm_sha1(pf), "factor_max_abs_diff": diff,
                  "factor_max_abs": scale,
                  "what": f"rank 0 factored the same n={n} matrix alone (nb={nb}) after the timed region; its own block columns of "
                          "the distributed factors are compared with the single-GPU factors (different GEMM kernels may serve "
                          "different local widths, so the factors agree to rounding, the pivots exactly)"}
            del F0
    except Exception as e:  # pragma: no cover
        p1 = {"error": repr(e)}
    barrier()
    del A, A0

    # ---- the previous round's workload, informational: weak-scaled LLT (n = 16384 N^(1/3)) on the same communicator ----
    also = {}
    try:
        nw = weak_n(world, DIST_NB)
        torch.manual_seed(1234)
        G = torch.randn((nw, nw), dtype=torch.float64, device=dev)
        gc = torch.as_tensor(lay.global_col_indices(nw, DIST_NB, world, rank), device=dev)
        S0 = (G @ G[gc, :].T)
        S0[gc, torch.arange(gc.numel(), device=dev)] += nw
        S0 = S0.T.contiguous().T
        del G
        S = S0.clone(memory_format=torch.preserve_format)

        def lstep():
            S.copy_(S0)
            fail, _ = lay.cholesky_in_place(S, nw, nb=DIST_NB)
            assert fail == -1
        lstep()
        barrier()
        a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for _ in range(3):
            lstep()
        a1.record(stream)
        barrier()
        tw = torch.tensor([a0.elapsed_time(a1) / 3], dtype=torch.float64, device=dev)
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        also["llt_weak"] = {"n": nw, "nb": DIST_NB, "ms_per_step": float(tw.item()), "value": llt_flops(nw) / (float(tw.item()) * 1e-3) / 1e12,
                            "unit": UNIT, "what": "weak-scaled LLT of round 1 (n^3 / (3 N) flop per GPU held at the n = 16384 value)"}
        del S, S0
    except Exception as e:  # pragma: no cover
        also["llt_weak"] = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"f64 partial-pivoting LU, ONE n={n} Gaussian matrix factored by {world} GPUs (BASELINE.json configs[2]; "
                                   f"1-D block-column-cyclic, nb={nb}, NCCL broadcast of panel + transpositions, look-ahead); strong "
                                   "scaling: same matrix and 2 n^3 / 3 flop for every N; step = restore copy + factor. The 1-GPU point "
                                   "of this curve is the `configs2_lu_n32768` block of the N = 1 line",
                       "n": n, "nb": nb, "layout": "column-major", "parallelism": f"block-column-cyclic x{world}",
                       "l2": f"inputs ({n * n * 8 / world / 1e9:.1f} GB per GPU) exceed the 126 MB L2; no flush needed",
                       "perm_sha1": r["perm_sha1"], "probe_residual": r["probe_residual"]},
            "clocks": r.get("clocks"), "e2e": e2e, "gpu_launches": r["launches"], "roofline": roof,
            "cpu_baseline": None, "p1_check": p1, "also": also,
        }
        print(json.dumps(line), flush=True)
    faer_b200.dist.finalize()
    dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=0, help="matrix dimension (default: 16384 at N=1, weak-scaled for N>1)")
    ap.add_argument("--nb", type=int, default=DIST_NB, help="block-column width of the distributed layout (N>1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the factor of the last one as DIR/<name>.npy (1-GPU arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1):
        ap.error("--dump-outputs needs the 1-GPU arm (--impl b200 --gpus 1)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist

    import faer_b200
    from faer_b200 import linalg as la

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = faer_b200.load()
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        faer_b200.dist.init_from_torch_distributed()
    lay = faer_b200.dist
    stream = torch.cuda.current_stream()
    lib.faer_b200_set_stream(stream.cuda_stream)
    if world > 1:
        return main_lu_strong(args, torch, dist, faer_b200, lay, lib, dev, stream, world, rank, local_rank)

    nb = args.nb
    n = args.n or N_DEFAULT
    distributed = False

    # ---- synthetic SPD input: A = G G^T + n I (same G on every rank); each rank keeps its block columns ----
    torch.manual_seed(1234)
    G = torch.randn((n, n), dtype=torch.float64, device=dev)
    if distributed:
        gcols = torch.as_tensor(lay.global_col_indices(n, nb, world, rank), device=dev)
        A0 = (G @ G[gcols, :].T)  # n x local_cols (row-major storage)
        A0[gcols, torch.arange(gcols.numel(), device=dev)] += n
        A0 = A0.T.contiguous().T  # column-major local matrix
    else:
        gcols = None
        A0 = torch.addmm(n * torch.eye(n, dtype=torch.float64, device=dev), G, G.T).T  # symmetric, column-major view
    del G
    A = A0.clone(memory_format=torch.preserve_format)

    def factor():
        if distributed:
            fail, _ = lay.cholesky_in_place(A, n, nb=nb)
            assert fail == -1
        else:
            la.cholesky_in_place(A)

    def step():
        A.copy_(A0)
        factor()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    launches0 = lib.faer_b200_launch_count()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    t_wall1 = time.time()
    my_launches = lib.faer_b200_launch_count() - launches0
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop(t_wall0, t_wall1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    # one factorisation of the (global) n x n matrix per step, whatever the number of ranks
    value = llt_flops(n) / (ms_per_step * 1e-3) / 1e12
    if args.dump_outputs:
        dump_llt_factor(torch, A, args.dump_outputs)

    # ---- correctness guard on the timed data (cheap probe): A x == L (L^T x), reduced over the ranks ----
    torch.manual_seed(99)
    x = torch.randn((n, 2), dtype=torch.float64, device=dev)
    if distributed:
        rows = torch.arange(n, device=dev)
        Lloc = torch.where(rows[:, None] >= gcols[None, :], A, torch.zeros((), dtype=torch.float64, device=dev))
        lhs = A0 @ x[gcols, :]
        rhs = Lloc @ (Lloc.T @ x)
        amax = A0.abs().max().reshape(1)
        dist.all_reduce(lhs); dist.all_reduce(rhs); dist.all_reduce(amax, op=dist.ReduceOp.MAX)
        resid = float((lhs - rhs).abs().max()) / (float(amax.item()) * n)
        del Lloc
    else:
        L = torch.tril(A)
        resid = float((A0 @ x - L @ (L.T @ x)).abs().max()) / (float(A0.abs().max()) * n)
        del L

    # ---- roofline of the dominant kernel (the DMMA GEMM doing the trailing updates), rank 0's view ----
    roof = None
    import ctypes as C
    # The profiled step runs the SAME block-column schedule with the two-stream look-ahead switched off: with look-ahead
    # the panel-chain GEMMs share the SMs with the trailing update, and per-launch event times of co-running kernels
    # overlap (their sum exceeds the step), which says nothing about the kernel. Serial launches give its own duration.
    A.copy_(A0)
    lib.faer_b200_profile_begin()
    fail, _ = lay.cholesky_in_place(A, n, nb=(nb if distributed else 256), lookahead=False)
    assert fail == -1
    barrier()
    flops = C.c_double(0); ms = C.c_double(0); cnt = C.c_ulonglong(0)
    lib.faer_b200_profile_end(C.byref(flops), C.byref(ms), C.byref(cnt))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "profiles", "r01_f64_peaks.json")))
    except Exception:
        pass
    peak = peaks.get("dmma_tflops_sustained", 36.9)
    ach = flops.value / (ms.value * 1e-3) / 1e12 if ms.value > 0 else None
    # DRAM traffic of the dominant kernel per launch: only from an ncu capture of THIS workload's launches (the SYRK-like
    # trailing updates of the n = 16384 LLT), profiles/r02_llt_gemm_traffic.json; null when that capture does not exist
    traffic = None
    traffic_src = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_llt_gemm_traffic.json")))
        traffic = tj.get("dram_bytes_per_launch")
        traffic_src = tj.get("source")
    except Exception:
        pass
    bf16 = None
    try:
        bf16 = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops_sustained")
    except Exception:
        pass
    roof = {"bound": "tensor", "kernel": "gemm_f64_ws_kernel / gemm_f64_kernel (DMMA.8x8x4 trailing updates: TMA-fed "
                                          "warp-specialised kernel for the large ones, cp.async kernel for the panel chain's)",
            "achieved": ach, "peak": peak,
            "unit": "TFLOP/s", "frac": (ach / peak) if ach else None, "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_bytes_per_launch": "16 (n-j)^2/2 + 16 (n-j) nb: lower half of dst read + written, the panel read twice",
            "launches_per_step": int(cnt.value), "ms_in_kernel_per_step": ms.value,
            "flops_in_kernel_per_step": flops.value,
            "peak_source": "measured on this pool: DMMA.8x8x4 issue-bound peak, profiles/r01_f64_peaks.json "
                           "(tcgen05 has no f64 kind; MEASURED_PEAKS.json only has bf16: "
                           f"{bf16} TF/s sustained => frac_of_bf16 = {(ach / bf16) if (ach and bf16) else None})",
            "how": "CUDA events around every launch of the kernel on the launching stream, one extra profiled step right "
                   "after the timed region (rank 0), same block-column schedule with the look-ahead overlap off so that "
                   "launches do not share the SMs; achieved = sum(algorithmic flop per launch) / sum(duration)"}

    # ---- e2e: same metric with HOST (pinned) buffers, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        rows_, cols_ = A0.shape
        hA0 = torch.empty((cols_, rows_), dtype=torch.float64, pin_memory=True)  # storage of the column-major matrix
        hA0.copy_(A0.T)
        hA = torch.empty((cols_, rows_), dtype=torch.float64, pin_memory=True)
        reps = max(2, min(args.steps, 3))
        bytes_h2d = rows_ * cols_ * 8
        if distributed:
            dA = torch.empty((cols_, rows_), dtype=torch.float64, device=dev)

            def e2e_call():
                dA.copy_(hA, non_blocking=True)            # H2D of this rank's block columns
                fail, _ = lay.cholesky_in_place(dA.T, n, nb=nb)
                hA.copy_(dA, non_blocking=True)            # D2H of the factor
                torch.cuda.synchronize()
                assert fail == -1
            how = "faer_b200.dist.cholesky_in_place on this rank's block columns, pinned host <-> device copies timed"
        else:
            hv = hA.numpy().T  # column-major view over pinned memory

            def e2e_call():
                la.cholesky_in_place(hv)  # H2D + factorisation + D2H inside the C-ABI call, synchronous
            # the call streams block columns (width 256) through the factorization: only the part on / below the
            # diagonal blocks crosses PCIe (the strict upper triangle is neither read nor written by LLT)
            # (the driver's block boundaries, csrc/dist.cu: llt_block_bounds — 256-wide, 128-wide in the last 6144 columns)
            bw = int(os.environ.get("FAER_B200_NB", "0")) or 256
            tail = int(os.environ.get("FAER_B200_LLT_TAIL", "6144"))
            bytes_h2d, j0 = 0, 0
            while j0 < n:
                w = min(128 if (bw > 128 and n - j0 <= tail) else bw, n - j0)
                bytes_h2d += (n - j0) * w * 8
                j0 += w
            how = ("libfaer_v0_23_llt_factor_in_place_f64 on a pinned HOST matrix (wall clock around the synchronous call); "
                   "block columns are uploaded / downloaded on copy streams while the factorization runs")
        hA.copy_(hA0); e2e_call()  # warm-up (pool allocation)
        ts = []
        for _ in range(reps):
            hA.copy_(hA0)
            barrier()
            t0 = time.perf_counter()
            e2e_call()
            ts.append(time.perf_counter() - t0)
        tt = torch.tensor([float(np.mean(ts))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": llt_flops(n) / float(tt.item()) / 1e12, "unit": UNIT,
               "h2d_bytes_per_step": bytes_h2d * world, "d2h_bytes_per_step": bytes_h2d * world,
               "ms_per_step": 1e3 * float(tt.item()), "how": how}
        if not distributed:
            # same probe as above on the factor that came back to the host (not timed)
            Lh = torch.tril(hA.to(dev).T)
            e2e["probe_residual"] = float((A0 @ x - Lh @ (Lh.T @ x)).abs().max()) / (float(A0.abs().max()) * n)
            del Lh
        del hA, hA0

    # ---- the other two numbers BASELINE.json's metric names (f64 GEMM and LU at the same n), device-resident, N = 1 only;
    # informational: `value` stays the LLT of configs[1] ----
    also = None
    if world == 1 and not args.no_e2e:
        def _best_ms(f, reps=2):
            f(); torch.cuda.synchronize(); best = 1e30
            for _ in range(reps):
                a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
                a0.record(stream); f(); a1.record(stream); torch.cuda.synchronize()
                best = min(best, a0.elapsed_time(a1))
            return best
        del A
        torch.manual_seed(4321)
        X = torch.randn((n, n), dtype=torch.float64, device=dev).T
        Y = torch.randn((n, n), dtype=torch.float64, device=dev).T
        Z = torch.empty((n, n), dtype=torch.float64, device=dev).T
        t_gemm = _best_ms(lambda: la.matmul(Z, la.Accum.Replace, X, Y, 1.0))
        del Y, Z
        Xw = X.clone(memory_format=torch.preserve_format)
        pf = torch.zeros(n, dtype=torch.int64, device=dev); pi = torch.zeros(n, dtype=torch.int64, device=dev)
        t_copy = _best_ms(lambda: Xw.copy_(X))

        def _lu():
            Xw.copy_(X)
            la.lu_in_place(Xw, pf, pi)
        t_lu = _best_ms(_lu) - t_copy
        also = {"gemm_f64_tflops": 2.0 * n ** 3 / t_gemm / 1e9, "gemm_ms": t_gemm,
                "lu_f64_tflops": 2.0 * n ** 3 / 3.0 / t_lu / 1e9, "lu_ms": t_lu, "n": n,
                "what": "device-resident f64 GEMM (Replace, alpha = 1) and partial-pivoting LU (u64 indices) at the same n"}
        del X, Xw
        # ---- the other BASELINE.json configs (f32 QR 65536 x 4096, bidiagonalization and c64 GEMM at n = 8192), timed by
        # tools/bench_other_configs.py in a CHILD process: informational, and nothing that happens there (not even an abort)
        # can touch this line's headline fields ----
        try:
            import subprocess
            child = subprocess.run([sys.executable, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools",
                                                                 "bench_other_configs.py")],
                                   capture_output=True, text=True, timeout=300)
            last = [ln for ln in child.stdout.strip().splitlines() if ln.startswith("{")]
            also["other_configs"] = json.loads(last[-1]) if last else {"error": f"exit {child.returncode}: {child.stderr[-300:]}"}
        except Exception as e:  # pragma: no cover
            also["other_configs"] = {"error": repr(e)}

    # ---- configs[2] at one GPU: the N = 1 point of the strong-scaling curve the N > 1 lines report (same matrix, same code) ----
    lu_block = None
    a0_gb = A0.numel() * 8 / 1e9
    if not args.no_e2e:
        try:
            del A0
            torch.cuda.empty_cache()
            r = run_lu(torch, dist, lay, lib, dev, stream, 1, 0, local_rank, LU_N, LU_NB, steps=3, warmup=1, sample_clocks=False)
            lu_block = {"workload": f"f64 partial-pivoting LU n={LU_N} (BASELINE.json configs[2]) on 1 GPU, nb={LU_NB}; "
                                    "step = restore copy + factor; same generator / seeds as the N > 1 lines",
                        "value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"], "steps": 3, "warmup": 1,
                        "perm_sha1": r["perm_sha1"], "probe_residual": r["probe_residual"], "gpu_launches": r["launches"]}
            del r
        except Exception as e:  # pragma: no cover
            lu_block = {"error": repr(e)}

    cpu = None
    proxy = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu, _, _ = cpu_llt_sample()
        proxy = lapack_proxy(min(n, 8192))

    if rank == 0:
        if distributed:
            wl = (f"f64 Cholesky LLT, ONE n={n} matrix factored by {world} GPUs (1-D block-column-cyclic, nb={nb}, NCCL panel "
                  f"broadcast + look-ahead); weak scaling of BASELINE.json configs[1] (n=16384 at N=1): n^3/(3N) flop per GPU held "
                  "constant; SPD = G G^T + n I; step = restore copy + factor")
        else:
            wl = f"f64 Cholesky LLT n={n} (BASELINE.json configs[1]); SPD = G G^T + n I; step = restore copy + factor"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl, "n": n, "layout": "column-major",
                       "parallelism": f"block-column-cyclic x{world}" if distributed else "single GPU",
                       "l2": f"inputs ({a0_gb:.1f} GB per GPU) exceed the 126 MB L2; no flush needed",
                       "probe_residual": resid},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(my_launches),
            "roofline": roof, "cpu_baseline": cpu, "cpu_lapack_proxy": proxy, "configs2_lu_n32768": lu_block, "also": also,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        faer_b200.dist.finalize()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
