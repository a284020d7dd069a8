#!/usr/bin/env python
"""bench.py — suggestions/sec at (N=8192 trials, M=1,048,576 candidates, D=32), Matérn-5/2 GP, EI  (BASELINE.json cfg 3).

One "step" = one full suggestion at fixed θ: Gram → Cholesky → L⁻¹/alpha → sweep of this rank's candidate rows (stratified
calibration rows, tensor-core K*, cta_group::2 ranking contraction, acquisition bounds, FP64 decision among the survivors) →
first-index argmax (→ one 32-byte-per-rank NCCL all-gather inside libkbo when N > 1).

  value     device-resident inputs, CUDA-event timed, max over ranks.
  e2e       the same through kbo_suggest_host: HOST buffers in (pinned), H2D + 32-byte D2H inside the timed region.
  roofline  the dominant kernel (tc_rank_kernel): algorithmic flops (rows·N² per launch) ÷ its mean launch time (CUDA events
            recorded around every launch inside libkbo) against the measured bf16 tensor peak; `kstar_hbm` the K* generation
            kernel against the measured HBM bandwidth; `acquisition_hbm` the standalone acquisition pass ("acquisition HBM
            GB/s vs peak").
  cpu_baseline / --impl reference   the oracle (fp64 NumPy/SciPy port of the sklearn path; scikit-optimize itself is not
            installable here) on all host cores: full N=8192 fit + 8192-row candidate batches (BASELINE.md §3.4), the sweep
            extrapolated linearly in M (it is linear).

Multi-GPU (torchrun, one rank per GPU): weak scaling — every rank runs the full N=8192 fit (replicated, bit-identical) and
sweeps its own 1,048,576-row shard of an R·1,048,576 grid; `value` counts R (N=8192, M=1M)-suggestion units per step and
`suggestions_per_s_actual` the suggestions over the R·M grid actually produced.  `other_configs` adds what BASELINE.json asks
beyond that: the SAME 1M grid split R ways (strong scaling) and, at R = 8, config 5 (one 16M grid, 2M rows per rank).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from kubeflow_b200 import workload as W   # noqa: E402  (the workload of record; no oracle import on the product arm)

N_TRIALS, M_CAND, DIM = 8192, 1_048_576, 32
KERNEL, ACQ = "matern52", "ei"
METRIC = "suggestions/sec at (N=8192, M=1M, D=32)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


def kernel_traffic(name, rows_per_launch):
    """dram bytes per launch from the committed `ncu --set full` capture of that kernel (profiles/), scaled by rows."""
    p = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(p):
        return None
    d = json.load(open(p))
    out = {"bytes_per_launch": (d["dram_read_bytes"] + d["dram_write_bytes"]) * rows_per_launch / d["rows"], "source": d["source"],
           "captured_rows_per_launch": d["rows"]}
    for k in ("algorithmic_bytes_per_launch", "ncu_tensor_pipe_active_pct_of_active", "ncu_dram_pct_of_peak", "ncu_l2_hit_pct", "ncu_l2_to_sm_bytes",
              "why_traffic_exceeds_algorithmic"):
        if k in d:
            out[k] = d[k] * rows_per_launch / d["rows"] if k in ("algorithmic_bytes_per_launch", "ncu_l2_to_sm_bytes") else d[k]
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(len(r) > col and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "power_w_median": float(np.median(pw)) if pw else None}


# ---------------------------------------------------------------------------------------------------------------------------
# CPU side: the oracle on the host cores (the only place bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------------------------------------
def _host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference(n_trials, dim, batches, rows_per_batch=8192, m_total=M_CAND):
    """Full fit at N = n_trials + `batches` candidate batches of `rows_per_batch` rows (BASELINE.md §3.4), on every host core —
    the BLAS/OpenMP pools are forced to the core count, so a launcher's OMP_NUM_THREADS=1 (torchrun sets it) cannot cripple
    it.  The sweep time is extrapolated linearly in M."""
    from threadpoolctl import threadpool_info, threadpool_limits
    from oracle import gp_oracle as O
    cores = _host_threads()
    with threadpool_limits(limits=cores):
        used = max([i.get("num_threads", 1) for i in threadpool_info()] + [1])
        rows = batches * rows_per_batch
        X, y, Xc = O.synthetic(n_trials, rows, dim)
        th = O.theta_of_record(dim)
        t0 = time.perf_counter()
        fit = O.gp_fit(X, y, kind=KERNEL, length_scale=th["length_scale"], amplitude=th["amplitude"], noise=th["noise"])
        t_fit = time.perf_counter() - t0
        t0 = time.perf_counter()
        mu, std = O.gp_predict(fit, Xc, batch=rows_per_batch)
        a = O.acquisition(mu, std, float(y.min()), ACQ, th["xi"], th["kappa"])
        _ = O.first_argmax(a)
        t_sweep = time.perf_counter() - t0
    t_full = t_fit + t_sweep * (m_total / rows)
    return {"value": 1.0 / t_full, "unit": "suggestions/s", "cores": int(used), "kind": "port",
            "sample": f"full fit N={n_trials} ({t_fit:.2f}s) + {batches} batch(es) of {rows_per_batch} candidates ({t_sweep:.2f}s) extrapolated linearly "
                      f"to M={m_total}; BLAS threads forced to {used} of {os.cpu_count()} host CPUs",
            "fit_s": t_fit, "sweep_sample_s": t_sweep, "host_cpus": os.cpu_count(), "seconds_per_suggestion": t_full}


def run_reference(args, rank, out_fd):
    if rank != 0:
        return
    # BASELINE.md §3.4 asks for 16 batches of 8192 rows: they are spread over the timed steps (each step pays the full fit, as
    # the reference does on every tell) so that the whole --steps/--warmup run ends within a few minutes
    per_step = max(1, min(4, math.ceil(16 / max(args.steps, 1))))
    for _ in range(args.warmup):   # warm-up: thread pools, page faults — a reduced sample, untimed
        cpu_reference(2048, args.dim, 1, rows_per_batch=1024, m_total=args.candidates)
    secs, last = [], None
    for _ in range(args.steps):
        last = cpu_reference(args.trials, args.dim, per_step, m_total=args.candidates)
        secs.append(last["seconds_per_suggestion"])
    t = float(np.mean(secs))
    line = {"metric": METRIC, "value": 1.0 / t, "unit": "suggestions/s", "impl": "reference",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": W.describe(args.trials, args.candidates, args.dim, args.gpus, KERNEL, ACQ), "kernel": KERNEL, "acq": ACQ,
                       "note": "CPU arm: one suggestion per step on the host cores whatever --gpus says (rank 0 only); ms_per_step is the "
                               "extrapolated time of a whole suggestion, the measured sample is in cpu_baseline.sample",
                       "batches_of_8192_rows_per_step": per_step, "batches_over_the_timed_steps": per_step * args.steps,
                       "warmup_note": "warm-up steps run a reduced sample (N=2048 fit + one 1024-row batch)"},
            "cpu_baseline": {k: last[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": 1.0 / t, "unit": "suggestions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    line["cpu_baseline"]["value"] = line["value"]
    _emit(out_fd, line)


# ---------------------------------------------------------------------------------------------------------------------------
def _claim_stdout():
    """stdout carries ONE JSON line.  Libraries write banners to file descriptor 1 behind Python's back (NCCL prints its version on
    the first communicator of a process): fd 1 is pointed at stderr for the whole run and the line goes to the saved descriptor."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def _emit(saved_fd, line: dict):
    os.write(saved_fd, (json.dumps(line) + "\n").encode())


def dump_outputs(path, results):
    """What each timed path returned to its caller in its last timed step — the suggestion: global candidate index, acquisition
    value, posterior mean and std — as DIR/<path>_<field>.npy, one float64 array of one element per field (the index is exact in
    float64).  The inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    os.makedirs(path, exist_ok=True)
    for name, best in results.items():
        for field in ("index", "value", "mu", "std"):
            np.save(os.path.join(path, f"{name}_{field}.npy"), np.array([getattr(best, field)], dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--trials", type=int, default=N_TRIALS)       # for quick local experiments only; the bench of record uses defaults
    ap.add_argument("--candidates", type=int, default=M_CAND)
    ap.add_argument("--dim", type=int, default=DIM)
    ap.add_argument("--var-mode", default="tc", choices=["tc", "f64"])
    ap.add_argument("--k-span", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the suggestion of the last timed step of the device and e2e paths to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    out_fd = _claim_stdout()
    if args.impl == "reference":
        run_reference(args, rank, out_fd)
        return

    import torch
    import torch.distributed as dist
    from kubeflow_b200.gp import GPEngine

    if args.warmup < 3:
        args.warmup = 3
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep NCCL's version banner off stdout: stdout carries ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    N, M, D = args.trials, args.candidates, args.dim
    th = W.theta_of_record(D)
    X, y = W.trials(N, D)
    Xc = W.candidates(M, D, offset=rank * M)   # this rank's shard of the R·M grid, fp32
    goff = rank * M

    eng = GPEngine(local, kernel=KERNEL, acq=ACQ, var_mode=args.var_mode, tc_k_span=args.k_span, **th)
    if world > 1:   # the exchange lives inside libkbo: one ncclAllGather of 32 bytes per rank (kbo_allreduce_argmax)
        box = [GPEngine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        eng.comm_init(world, rank, box[0])
    Xd, yd, Xcd = torch.tensor(X, device=dev), torch.tensor(y, device=dev), torch.tensor(Xc, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step, steps, warmup):
        """W untimed + K timed steps, barrier + synchronize on both sides, CUDA events, max over ranks -> ms per step."""
        out = None
        for _ in range(warmup):
            out = step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = step()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps, out

    def step_device():
        eng.tell(Xd, yd)
        return eng.ask(Xcd, global_offset=goff, allreduce=world > 1)

    # ---- device-resident value ---------------------------------------------------------------------------------
    sampler = ClockSampler(local)
    for _ in range(args.warmup):
        best = step_device()
    barrier()
    if rank == 0:
        sampler.start()
    ms_step, best = timed(step_device, args.steps, 0)
    survivors, rank_err, rank_mu_err, unrefined = eng.last_contenders(), eng.last_rank_error(), eng.last_rank_mu_error(), eng.last_unrefined()

    # ---- end to end: host buffers through kbo_suggest_host (the exchange is inside the call when N > 1) ---------------
    Xp, yp = torch.tensor(X).pin_memory(), torch.tensor(y).pin_memory()
    Xcp = torch.tensor(Xc).pin_memory()
    Xh, yh, Xch = Xp.numpy(), yp.numpy(), Xcp.numpy()
    tims = []

    def step_host():
        b, t = eng.suggest_host(Xh, yh, Xch, global_offset=goff)
        tims.append(t)
        return b

    ms_step_e2e, best_h = timed(step_host, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    tims = tims[-args.steps:]
    assert best_h.index == best.index, "host and device paths disagree on the argmax"
    if args.dump_outputs and rank == 0:   # after the exchange every rank holds the same global suggestion
        dump_outputs(args.dump_outputs, {"device": best, "e2e": best_h})
    chunks = tims[-1]["chunks"]
    launches = sum(t["launches"] for t in tims)
    mean = lambda k: float(np.mean([t[k] for t in tims]))   # noqa: E731

    # ---- standalone acquisition pass: the HBM-bound kernel (8 B/candidate in + 4 B out), at this rank's M and at cfg5's 16M ----
    flush64 = torch.zeros((256 << 20) // 8, dtype=torch.int64, device=dev)   # > 126 MB L2
    flush_sink = torch.zeros((), dtype=torch.int64, device=dev)

    def acq_bw(Ma):
        mu_n = torch.randn(Ma, device=dev, dtype=torch.float32)
        var_n = torch.rand(Ma, device=dev, dtype=torch.float32)
        acq_o = torch.empty(Ma, device=dev, dtype=torch.float32)
        ts = []
        for i in range(10):
            # evict with READS of a 256 MiB buffer: a write-based flush leaves ~126 MB of dirty L2 lines whose write-back then
            # competes with the timed kernel for DRAM bandwidth
            flush_sink.copy_(flush64.sum())
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            eng.lib.kbo_acq_argmax(eng._h, mu_n.data_ptr(), var_n.data_ptr(), Ma, 0, 0, 0.0, 1.0, -1.0, 0.01, 1.96, acq_o.data_ptr(),
                                   eng._best_dev.data_ptr(), eng._stream())
            a1.record()
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(a0.elapsed_time(a1))
        t = float(np.median(ts))
        return 12.0 * Ma / (t * 1e-3) / 1e9, t

    acq_gbs, acq_launch_ms = acq_bw(M)
    acq_gbs16, acq_launch_ms16 = acq_bw(16_777_216)

    # ---- the tensor-core kernel of record, measured on the FULL contraction (kbo_set_rank_prefix(h, 0)): the product path's
    # pruning pass runs the same kernel over the first eighth of the trial tiles only, which is too short a launch to rate ----
    prefix_survivors = eng.last_prefix_survivors()
    full_tims = []
    if args.var_mode == "tc" and rank == 0:
        e_full = GPEngine(local, kernel=KERNEL, acq=ACQ, var_mode="tc", rank_prefix=0, tc_k_span=args.k_span, **th)
        for i in range(5):
            b_full, t_full = e_full.suggest_host(Xh, yh, Xch, global_offset=goff)
            if i >= 2:
                full_tims.append(t_full)
        assert b_full.index == (best.index if world == 1 else b_full.index)
        e_full.close()

    other = {}
    # ---- multi-GPU: the same 1M grid split R ways (strong scaling) and, at R = 8, BASELINE.json config 5 ----------------------
    if world > 1 and not args.no_extras:
        from kubeflow_b200.dist import shard_rows
        lo, hi = shard_rows(M, rank, world)
        Xs_d = torch.tensor(W.candidates(hi - lo, D, offset=lo), device=dev)
        ms_s, b_s = timed(lambda: (eng.tell(Xd, yd), eng.ask(Xs_d, global_offset=lo, allreduce=True))[1], 3, 2)
        other["strong_scaling_M1M_grid"] = {"grid_candidates": M, "rows_per_rank": hi - lo, "ms_per_step": ms_s, "suggestions_per_s_actual": 1e3 / ms_s,
                                            "argmax_index": b_s.index, "argmax_value": b_s.value,
                                            "note": "the single-GPU workload's grid split over the ranks; the N=8192 FP64 fit is replicated on every rank (the Amdahl term)"}
        del Xs_d
        if world == 8:
            M5 = 16_777_216 // world
            X5_d = torch.tensor(W.candidates(M5, D, offset=rank * M5), device=dev)
            ms_5, b_5 = timed(lambda: (eng.tell(Xd, yd), eng.ask(X5_d, global_offset=rank * M5, allreduce=True))[1], 3, 2)
            other["cfg5_gp_ei_grid_16M_over_8_gpus"] = {"grid_candidates": 16_777_216, "rows_per_rank": M5, "ms_per_step": ms_5,
                                                        "suggestions_per_s_actual": 1e3 / ms_5, "argmax_index": b_5.index, "argmax_value": b_5.value}
            del X5_d

    # ---- single GPU extras: the three-product sweep and a flat landscape beside the headline, the other BASELINE configs ----------
    if rank == 0 and full_tims:
        other["full_ranking_pass"] = {"ms_per_step_e2e": float(np.mean([t["total_ms"] for t in full_tims])),
                                      "variance_kernel_ms": float(np.mean([t["var_kernel_ms"] for t in full_tims])),
                                      "kstar_kernel_ms": float(np.mean([t["cross_kernel_ms"] for t in full_tims])),
                                      "note": "kbo_set_rank_prefix(h, 0): no pruning pass — tensor-core K* and cta_group::2 contraction over the whole grid "
                                              "(also what a landscape too flat to prune costs, before any three-product redo)"}
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            e3 = GPEngine(local, kernel=KERNEL, acq=ACQ, var_mode="tc", tc_fast=False, **th)
            ms_3, b_3 = timed(lambda: (e3.tell(Xd, yd), e3.ask(Xcd))[1], 2, 1)
            other["three_product_sweep"] = {"ms_per_step": ms_3, "suggestions_per_s": 1e3 / ms_3, "argmax_index": b_3.index, "argmax_value": b_3.value,
                                            "fp64_refined_contenders": e3.last_contenders(),
                                            "note": "kbo_set_tc_fast(h, 0): FP64 K* kernel + fp16x3 contraction over the whole grid — what a caller asking "
                                                    "for per-candidate arrays gets, and the fallback when the ranking pass cannot prune"}
            e3.close()
            # a landscape nothing can prune: all candidates in a 1e-4 cube next to the incumbent (EI positive, flat to ~1e-6) -> the prefix
            # bound keeps everything -> full ranking pass -> > 4096 survivors -> three-product redo -> window narrowing; reported so the
            # headline's dependence on a peaked EI is visible
            flat = torch.tensor(np.clip(X[int(np.argmin(y))] + 0.02 + 1e-4 * (np.random.default_rng(5).random((M, D)) - 0.5), 0, 1).astype(np.float32), device=dev)
            ms_f, b_f = timed(lambda: (eng.tell(Xd, yd), eng.ask(flat))[1], 2, 1)
            other["flat_landscape"] = {"ms_per_step": ms_f, "suggestions_per_s": 1e3 / ms_f, "kept_by_the_pruning_pass": eng.last_prefix_survivors(),
                                       "survivors_of_the_ranking_pass": eng.last_contenders(),
                                       "decision": {0: "fp64 among all survivors", 1: "fp64 among the best 4096 by fp32 value", 2: "not refined"}[eng.last_unrefined()],
                                       "argmax_value": b_f.value}
            del flat
            X2, y2 = W.trials(1024, 8)
            Xc2 = W.candidates(65536, 8)
            e2 = GPEngine(local, kernel="rbf", acq="ei", var_mode="auto", **W.theta_of_record(8))
            X2d, y2d, Xc2d = torch.tensor(X2, device=dev), torch.tensor(y2, device=dev), torch.tensor(Xc2, device=dev)
            ms_2, b2 = timed(lambda: (e2.tell(X2d, y2d), e2.ask(Xc2d))[1], 10, 3)
            other["cfg2_gp_rbf_n1024_m65536_d8"] = {"suggestions_per_s": 1e3 / ms_2, "var_mode": "auto (FP64 contraction)", "argmax_index": b2.index}
            e2.close()
            from kubeflow_b200.cmaes import CmaEs
            es = CmaEs(np.full(128, 3.0), 2.0, popsize=4096, seed=7, device=local)
            es.run_synthetic("rastrigin", 20)
            r4 = es.run_synthetic("rastrigin", 200)
            other["cfg4_cmaes_d128_pop4096_200gen"] = {"generations_per_s": r4["generations_per_s"], "elapsed_ms": r4["elapsed_ms"],
                                                        "jacobi_sweeps_last": r4["jacobi_sweeps"]}
            es.close()
            other["grpc_cfg3_request"] = grpc_cfg3_request(local, X, y, N, M, D)
        except Exception as e:  # noqa: BLE001 — the extras must never take the headline line down
            other["error"] = f"{type(e).__name__}: {e}"

    if rank == 0:
        pk = peaks()
        fast_rank = args.var_mode == "tc" and rank_err > 0.0
        rank_tc = fast_rank and rank_mu_err > 0.0
        pruned = rank_tc and 1 <= prefix_survivors <= 16384
        fmean = (lambda k: float(np.mean([t[k] for t in full_tims]))) if full_tims else mean
        fchunks = full_tims[-1]["chunks"] if full_tims else chunks
        rows_per_launch = M / max(fchunks, 1)
        var_launch_ms = fmean("var_kernel_ms") / max(fchunks, 1)
        cross_launch_ms = mean("cross_kernel_ms") / max(chunks, 1)
        flops_launch = rows_per_launch * float(N) * float(N)           # Σ_j Σ_{k<=j} 2 flops = N² per candidate row
        achieved_tf = flops_launch / (var_launch_ms * 1e-3) / 1e12
        mma_products = 1.0 if fast_rank else 3.0
        # FP64 flops of the fit: Cholesky N³/3; the lazy inverse (default when the sweep prunes) adds only the leading rows of L⁻¹
        # the pruning pass contracts with (lead³/3) and two triangular solves; a full inverse adds N³/3
        lazy_fit = bool(pruned)
        lead = min(N, 512 * ((((N + 255) // 256 + 1) // 2 + 7) // 8))
        fit_flops = N ** 3 / 3.0 + (lead ** 3 / 3.0 + 4.0 * N * N if lazy_fit else N ** 3 / 3.0)
        fit_tflops = fit_flops / (mean("fit_ms") * 1e-3) / 1e12
        fp64_peak = eng.fp64_peak_tflops()
        kernel = "tc_rank_kernel" if rank_tc else ("tc_variance_pair_kernel" if os.environ.get("KBO_TC_PAIR", "1") != "0" else "tc_variance_kernel")
        Npad = (N + 255) // 256 * 256
        kstar_bytes = rows_per_launch * Npad * 2.0
        line = {
            "metric": METRIC, "value": world * 1e3 / ms_step, "unit": "suggestions/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "suggestions_per_s_actual": 1e3 / ms_step,
            "dtype": ("f64 fit / ranking pass: fp16 hi+lo tcgen05 dot products -> fp32 kernel values -> fp16 K* plane, fp16 cta_group::2 contraction "
                      "(fp32 accumulate), fp32 mean / FP64 K*, mean and variance for the calibration rows and the survivors that decide"
                      if rank_tc else "f64 fit+mean / fp16 tcgen05 ranking pass over sigma² (1 product, fp32 accumulate) + FP64 decision among the survivors"
                      if fast_rank else "f64 fit+mean / fp16x3-split tcgen05 variance (fp32 accumulate)") if args.var_mode == "tc" else "f64",
            "data": "synthetic",
            "config": {"workload": W.describe(N, M, D, world, KERNEL, ACQ),
                       "kernel": KERNEL, "acq": ACQ, "per_gpu_candidates": M, "grid_candidates": world * M, "var_mode": args.var_mode,
                       "l2": "inputs larger than L2 (Xc 128 MiB, W plane 128 MiB, K* scratch 4 GiB per chunk)",
                       "argmax_index": best.index, "argmax_value": best.value, "argmax_mu": best.mu, "argmax_std": best.std,
                       "survivors_decided_in_fp64": survivors, "decision": unrefined,
                       "pruning_pass": ({"prefix_of_trial_tiles": "first eighth (1/64 of the contraction's MMAs)", "candidates_kept": prefix_survivors,
                                         "pruned": bool(pruned)} if rank_tc else None),
                       "ranking_pass": ({"variance_error_on_calibration_rows": rank_err, "mean_error_on_calibration_rows": rank_mu_err,
                                         "calibration": "stratified rows i*M/n, n = 9472, through the FP64 K* kernel + three-product contraction; bounds = 8 x max error"}
                                        if fast_rank else None)},
            "e2e": {"value": world * 1e3 / ms_step_e2e, "unit": "suggestions/s", "ms_per_step": ms_step_e2e,
                    "h2d_bytes_per_step": int(X.nbytes + y.nbytes + Xc.nbytes), "d2h_bytes_per_step": 32,
                    "suggestions_per_s_actual": 1e3 / ms_step_e2e},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": kernel, "achieved": achieved_tf, "peak": pk["tf_sus"], "unit": "TFLOP/s",
                         "frac": achieved_tf / pk["tf_sus"], "peak_source": f"bf16_tflops_sustained, {pk['src']}",
                         "frac_of_burst_peak": achieved_tf / pk["tf_burst"],
                         "issued_mma_tflops": mma_products * achieved_tf * (1.0 + 256.0 / N), "mma_products_per_term": mma_products,
                         "traffic": kernel_traffic("tcrank_traffic.json" if rank_tc else "tcvar_traffic.json", rows_per_launch) if (rank_tc or not fast_rank) else None,
                         "launch_ms": var_launch_ms, "launches_per_step": chunks, "flops_per_launch": flops_launch,
                         "launch_note": "variance phase time / chunks (CUDA events inside libkbo around tc_rank_kernel + its 6 µs finish kernel)",
                         "share_of_step": {"note": "where the product path's step goes (phases_ms / ms_per_step); this object rates the kernel that carries "
                                                   "the path's M·N² term, which the pruning pass shrinks to 1/64 — the step's largest kernels are rated in "
                                                   "fit_fp64 (dgemm64_kernel, FP64 DMMA) and kstar_hbm / profiles (tc_kstar_kernel, MUFU-bound)",
                                           "fit": mean("fit_ms") / ms_step, "kstar_kernel": mean("cross_kernel_ms") / ms_step,
                                           "prefix_contraction_this_kernel": mean("var_kernel_ms") / ms_step, "calibration": mean("calib_ms") / ms_step,
                                           "bounds_and_fp64_decision": mean("acq_kernel_ms") / ms_step},
                         "measured_on": ("the full contraction, kbo_set_rank_prefix(h, 0), 3 steps through kbo_suggest_host in this run (%.1f ms per step): the product "
                                         "path above prunes with the same kernel over the first eighth of the trial tiles (%.2f ms per step) and contracts fully only "
                                         "the %d candidates that survive" % (fmean("total_ms"), mean("var_kernel_ms"), prefix_survivors)) if pruned else "the product path"},
            "fit_fp64": {"bound": "tensor (FP64 DMMA)", "kernels": "dgemm64_kernel (DMMA m8n8k4) + potf2_inv / trsm_panel chain on its own SM partition",
                         "flops": fit_flops, "ms": mean("fit_ms"), "achieved": fit_tflops, "peak": fp64_peak, "unit": "TFLOP/s", "frac": fit_tflops / fp64_peak,
                         "peak_source": "measured in this run: DMMA m8n8k4 on register operands, one 256-thread CTA per SM (kbo_debug_fp64_peak; "
                                        "MEASURED_PEAKS.json has no FP64 entry)",
                         "inverse": "lazy: leading %d rows of L^-1 + two panel solves" % lead if lazy_fit else "full",
                         "note": "the step's largest phase; FP64 by contract (fp32 Cholesky / alpha move EI by up to 4e-4). The trailing updates run at "
                                 "~24 TFLOP/s (K = 256 GEMMs, tests/studies/dgemm_probe.cu); the rest of the gap is the dependent chain of 128 "
                                 "single-CTA diagonal blocks, which the second half of the factorisation waits on"},
            "kstar_hbm": {"bound": "hbm", "kernel": "tc_kstar_kernel" if rank_tc else "cross_mean_kernel", "bytes_per_launch": kstar_bytes,
                          "launch_ms": cross_launch_ms, "achieved": kstar_bytes / (cross_launch_ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                          "frac": kstar_bytes / (cross_launch_ms * 1e-3) / 1e9 / pk["hbm"],
                          "note": "algorithmic bytes = the fp16 K* plane written once (rows x Npad x 2 B); the kernel is MUFU/issue-bound (2 MUFU + ~15 "
                                  "instructions per pair), not bandwidth-bound — profiles/r9_tckstar_cfg3_summary.csv"},
            "acquisition_hbm": {"kernel": "acq_kernel<float>", "bytes_per_candidate": 12, "candidates": M, "achieved": acq_gbs, "peak": pk["hbm"],
                                "unit": "GB/s", "frac": acq_gbs / pk["hbm"], "peak_source": f"hbm_gbs, {pk['src']}", "launch_ms": acq_launch_ms,
                                "at_16M_candidates": {"achieved": acq_gbs16, "frac": acq_gbs16 / pk["hbm"], "launch_ms": acq_launch_ms16},
                                "l2": "evicted by reading a 256 MiB buffer before each timed launch (clean lines: no write-back during the timed kernel)"},
            "other_configs": other,
            "phases_ms": {"fit": mean("fit_ms"), "calibration": mean("calib_ms"), "kstar_kernel": mean("cross_kernel_ms"),
                          "variance_kernel": mean("var_kernel_ms"), "acquisition_and_fp64_decision": mean("acq_kernel_ms"),
                          "h2d_candidates": mean("h2d_ms")},
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = {k: v for k, v in cpu_reference(N, D, 2, m_total=M).items() if k != "seconds_per_suggestion"}
        _emit(out_fd, line)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def grpc_cfg3_request(local, X, y, N, M, D):
    """The reference-facing surface at cfg3 scale: a real gRPC GetSuggestions carrying all finished trials as strings."""
    import grpc
    from kubeflow_b200.suggestion import api_pb as api
    from kubeflow_b200.suggestion.server import SuggestionStub, serve
    from kubeflow_b200.suggestion.service import SkoptService
    skopt_svc = SkoptService({"device": local})
    server, port = serve(skopt_svc, port=0, host="127.0.0.1")
    ch = grpc.insecure_channel(f"127.0.0.1:{port}", options=[("grpc.max_send_message_length", 1 << 28), ("grpc.max_receive_message_length", 1 << 28)])
    stub = SuggestionStub(ch)
    ex = api.Experiment()
    ex.name = "bench-cfg3"
    ex.spec.objective.type = api.MINIMIZE
    ex.spec.objective.objective_metric_name = "loss"
    ex.spec.algorithm.algorithm_name = "bayesianoptimization"
    for k_, v_ in {"n_initial_points": 0, "acq_func": "EI", "acq_optimizer": "sampling", "random_state": 1, "n_points": M, "var_mode": "tc"}.items():
        st_ = ex.spec.algorithm.algorithm_settings.add()
        st_.name, st_.value = k_, str(v_)
    for d_ in range(D):
        ps_ = ex.spec.parameter_specs.parameters.add()
        ps_.name, ps_.parameter_type = f"x{d_}", api.DOUBLE
        ps_.feasible_space.min, ps_.feasible_space.max = "0", "1"
    rq = api.GetSuggestionsRequest(experiment=ex, current_request_number=1)

    def add_trial(i, xs, yv):
        t_ = rq.trials.add()
        t_.name = f"t{i}"
        t_.spec.objective.objective_metric_name = "loss"
        t_.status.condition = api.SUCCEEDED
        for d_ in range(D):
            a_ = t_.spec.parameter_assignments.assignments.add()
            a_.name, a_.value = f"x{d_}", repr(float(xs[d_]))
        m_ = t_.status.observation.metrics.add()
        m_.name, m_.value = "loss", repr(float(yv))

    for i in range(N - 3):
        add_trial(i, X[i], y[i])
    calls = []
    for c_ in range(4):
        t0 = time.perf_counter()
        stub.GetSuggestions(rq)
        calls.append((time.perf_counter() - t0) * 1e3)
        add_trial(N - 3 + c_, X[min(N - 3 + c_, N - 1)], y[min(N - 3 + c_, N - 1)])
    out = {"trials_in_request": N, "request_bytes": rq.ByteSize(), "n_points": M, "cold_call_ms": calls[0],
           "steady_call_ms": float(np.median(calls[1:])), "ingest_last_call": skopt_svc.last_ingest,
           "engine_update_last_call": getattr(skopt_svc._services["bench-cfg3"].skopt_optimizer, "last_fit", None),
           "note": "in-process grpc.server, all finished trials resent as strings on every call; steady = one new trial per call"}
    ch.close()
    server.stop(0)
    return out


if __name__ == "__main__":
    main()
