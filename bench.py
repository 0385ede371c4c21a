#!/usr/bin/env python
"""Benchmark of the phys-optim hot path (BASELINE.json metric: optimised frames/sec of the batched staged
physics optimisation) and of the other two BASELINE configurations.

    python bench.py --gpus N --steps K --warmup W            # product arm (hand-written sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the oracle port of the reference algorithm
    python bench.py --workload long | contact ...             # BASELINE configs[4] / configs[2], same line schema

Default workload (`phys`): one "step" = one full staged solve (stages 1.1, 1.2, 2.1, 2.2, 3 and -- only for sequences
whose stage 3 did not succeed -- 4 of phys_optim.cpp:554-749) of a batch of synthetic 120-frame / 2-end-effector
sequences: BASELINE.json configs[1], batch 64 on one B200; 64 per GPU under torchrun (weak scaling, sequences are
independent NLPs; sharding, the solve, the device-side sampling into the send buffer and the one NCCL gather go through
the product's `chd.parallel.ShardedSolver`).  At 8 GPUs the named configuration of BASELINE.json configs[3]
(1024 sequences = 128 per GPU) is timed as well and reported under `named_config_1024`.

value : whole-job frames/s with the problem tables already resident in HBM (device-side reset of the iterate).
e2e   : the same metric through the public host API with host buffers: layout build + H2D + solve + gather + D2H of
        the solved trajectories inside the timed region.
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCHEDULE = "1.1,1.2,2.1,2.2,3,(4 if 3 failed)"
WORKLOADS = {
    # name: (frames, n_ee, dense, per-GPU batch, description)
    "phys": (120, 2, False, 64, "batch %d synthetic 120-frame sequences, 2 foot end-effectors, staged phys-optim (" + SCHEDULE + ")"),
    "long": (600, 4, True, None, "long-horizon: %d x 600-frame sequences, 4 end-effectors (toes + heels), dense contact phase switches, staged phys-optim (" + SCHEDULE + ")"),
}
STAGE_NAMES = ["1.1", "1.2", "2.1", "2.2", "3", "4"]


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.reasons, self.stop_flag = gpu, [], set(), False
        self.max_mhz = None

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def result(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------ CPU arm ------------
def _oracle_solve_one(task):
    seed, frames, n_ee, dense = task
    import chd
    from oracle.phys import OracleProblem
    p = chd.synth.make_problem(seed, frames, n_ee, dense=dense)
    t0 = time.perf_counter()
    o = OracleProblem(p)
    r = o.solve()
    dt = time.perf_counter() - t0
    res = {k: (s["status"], s["iters"], s["E0"], s["viol"], s["dual"]) for k, s in zip(r["stage_ids"], r["stages"])}
    return dt, res, r["success"]


def cpu_arm(seeds, cores, frames, n_ee, dense):
    """Times the CPU oracle (a port of the reference algorithm, NOT TOWR/ifopt/IPOPT/MA57) on the given sequences
    spread over `cores` processes (one sequence at a time per process, longest-first not known a priori).
    Returns frames/s, wall seconds, per-stage residual summary."""
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(cores) as pool:
        res = list(pool.imap_unordered(_oracle_solve_one, [(s, frames, n_ee, dense) for s in seeds], chunksize=1))
    wall = time.perf_counter() - t0
    return len(seeds) * frames / wall, wall, residual_summary_cpu(res)


def residual_summary_cpu(res):
    out = {}
    for k in STAGE_NAMES:
        rows = [r[1][k] for r in res if k in r[1]]
        if rows:
            out[k] = {"sequences": len(rows), "ok_frac": float(np.mean([r[0] == 0 for r in rows])),
                      "iters_mean": float(np.mean([r[1] for r in rows])), "iters_max": int(max(r[1] for r in rows)),
                      "max_nlp_error": float(max(r[2] for r in rows)), "max_constr_viol": float(max(r[3] for r in rows)),
                      "max_dual_inf": float(max(r[4] for r in rows))}
    out["success_frac"] = [float(np.mean([r[2][0] for r in res])), float(np.mean([r[2][1] for r in res]))]
    return out


def workload_config(name, world, per_gpu):
    frames, n_ee, dense, _, desc = WORKLOADS[name]
    return {"workload": desc % (per_gpu * world), "sequences": per_gpu * world, "frames": frames, "n_ee": n_ee,
            "per_gpu_batch": per_gpu, "seeds": "numpy default_rng(seed), seeds 0..sequences-1 (chd.synth.make_problem)",
            "l2": "256 MiB flush buffer written before every timed step (product arm)"}


def run_reference(args, rank, world, per_gpu):
    """`--impl reference`: the reference's algorithm on the host cores (the oracle port), all cores loaded.  The K steps
    run back to back through one process pool: every step is a bounded sample of the workload (same generator, its own
    seeds), sized from a one-sequence calibration so that the whole run takes about `--cpu-budget` seconds."""
    if rank != 0:
        return
    frames, n_ee, dense, _, _ = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    t_cal, _, _ = _oracle_solve_one((10_000, frames, n_ee, dense))                       # calibration sequence (not counted)
    steps = max(1, args.steps)
    per_step = int(max(1, min(per_gpu * world, round(cores * args.cpu_budget / (steps * max(t_cal, 1e-3) * 1.5)))))
    if per_step * steps < cores:                                                          # never leave cores idle
        per_step = -(-cores // steps)
    seeds = list(range(per_step * steps))
    v, wall, resid = cpu_arm(seeds, cores, frames, n_ee, dense)
    sample = ("%d steps x %d sequences x %d frames (seeds 0..%d of the workload's generator) through one pool of %d processes, "
              "one sequence per process at a time, %.1f s wall in total" % (steps, per_step, frames, len(seeds) - 1, cores, wall))
    line = {"impl": "reference", "metric": "optimised frames/sec (batched phys-optim)", "value": v, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.workload, world, per_gpu),
            "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "residual": resid,
            "note": "CPU arm = our C++ restatement of the reference NLP + the same interior-point algorithm (oracle/), NOT the reference's "
                    "TOWR/ifopt/IPOPT/MA57 stack, which cannot be built offline (DESIGN.md); speed-ups over this arm are 'vs in-repo port'"}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ product arm --------
def residual_summary_gpu(stats, sstat, siter, success):
    """stats (6,B,4), sstat / siter (6,B)"""
    out = {}
    for s, k in enumerate(STAGE_NAMES):
        ran = sstat[s] != -9
        if ran.any():
            out[k] = {"sequences": int(ran.sum()), "ok_frac": float((sstat[s][ran] == 0).mean()),
                      "iters_mean": float(siter[s][ran].mean()), "iters_max": int(siter[s][ran].max()),
                      "max_nlp_error": float(stats[s][ran, 1].max()), "max_constr_viol": float(stats[s][ran, 2].max()),
                      "max_dual_inf": float(stats[s][ran, 3].max())}
    out["success_frac"] = [float(success[:, 0].mean()), float(success[:, 1].mean())]
    return out


def time_solver(solver, steps, warmup, flush, barrier, torch):
    """W untimed + K timed resident steps (device-side reset, staged solve, device sampling, the one gather)."""
    last = None

    def step():
        flush.zero_()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = solver.solve(resident=True)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3, out

    for _ in range(warmup):
        step()
    barrier()
    l0 = solver.batch.launch_count()
    ts, per = [], []
    for _ in range(steps):
        dt, last = step()
        ts.append(dt)
        per.append(dict(solver.last_ms))
    barrier()
    return ts, last, solver.batch.launch_count() - l0, per


DUMP_LIMIT = 64 * 1024 * 1024
DUMP_SEQ_AXIS = {"samples": 0, "frames": 0, "success": 0, "stage_status": 1, "stage_iters": 1}


def dump_outputs(out, path):
    """Writes the arrays `ShardedSolver.solve` returned (sampled trajectories, per-sequence status) as <path>/<name>.npy in
    float64, in the caller's layout, so that two builds can be compared output for output.  Above DUMP_LIMIT bytes every
    array keeps the same fixed, seeded sample of sequences, whose indices go to sequence_index.npy.
    Compare with tolerances: the kernels accumulate with fp64 atomics, so two runs of one build already differ.  On a B200,
    64 x 120-frame sequences, two runs differed by ~1e-9 m / 1e-6 N per sequence, and by 2e-4 m / 2e-2 N in the one
    sequence whose stage-3 iteration count changed (the tolerances of tests/test_phys_gpu.py allow 5e-3 m / 5 N)."""
    arrays = {k: np.asarray(out[k], dtype=np.float64) for k in DUMP_SEQ_AXIS}
    n = arrays["frames"].shape[0]
    keep = int(DUMP_LIMIT // (sum(a.nbytes for a in arrays.values()) / n + 8))
    if keep < n:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: np.take(a, idx, axis=DUMP_SEQ_AXIS[k]) for k, a in arrays.items()}
        arrays["sequence_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def run_contact(args):
    """BASELINE.json configs[2] (contact-net inference, 100k windows, 1 B200): scripts/bench_contact.py emits the line."""
    cmd = [sys.executable, os.path.join(ROOT, "scripts", "bench_contact.py"), "--steps", str(args.steps), "--warmup", str(args.warmup)]
    if args.impl == "reference":
        cmd.append("--reference")
    sys.exit(subprocess.call(cmd))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="chd")
    ap.add_argument("--workload", default="phys", choices=["phys", "long", "contact"])
    ap.add_argument("--per-gpu", type=int, default=0, help="sequences per GPU (default: 64 for phys, 128 / GPUs for long)")
    ap.add_argument("--cpu-budget", type=float, default=150.0, help="seconds of wall clock the CPU arm aims for")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-named", action="store_true", help="skip the 1024-sequence pass at 8 GPUs")
    ap.add_argument("--named-world", type=int, default=8, help="world size at which the 128-per-GPU pass runs (8 = BASELINE configs[3])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float64, at most 64 MiB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload == "contact" or args.impl == "reference"):
        ap.error("--dump-outputs writes the product arm's phys-optim results (--workload phys or long)")
    rank, world, local = _env_int("RANK", 0), _env_int("WORLD_SIZE", 1), _env_int("LOCAL_RANK", 0)
    if args.workload == "contact":
        if rank == 0:
            run_contact(args)
        return
    frames, n_ee, dense, per_gpu_default, _ = WORKLOADS[args.workload]
    per_gpu = args.per_gpu or per_gpu_default or max(1, 128 // world)
    if args.impl == "reference":
        run_reference(args, rank, world, per_gpu)
        return
    import torch
    import torch.distributed as dist
    import chd
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(v):
        t = torch.tensor(v, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.cpu().numpy()

    def measure(per_gpu_b, steps, warmup, with_kernels):
        N = per_gpu_b * world
        problems = [chd.synth.make_problem(s, frames, n_ee, dense=dense) for s in range(N)]
        solver = chd.parallel.ShardedSolver(problems, device=local, rank=rank, world=world)
        ts, last, launches, per = time_solver(solver, steps, warmup, flush, barrier, torch)
        t_total = float(reduce_max([sum(ts)])[0])
        b = solver.batch
        res = {"N": N, "t_total": t_total, "launches": launches, "last": last, "solver": solver, "problems": problems,
               "solve_ms": float(np.mean([p["solve_ms"] for p in per])), "gather_ms": float(np.mean([p["gather_ms"] for p in per]))}
        # per-rank view: slowest sequence of the shard, local solve / gather time
        it_local = last["stage_iters"][:, solver.mine].sum(axis=0)
        mine = [int(rank), int(it_local.max()), float(it_local.mean()), res["solve_ms"], res["gather_ms"]]
        if world > 1:
            allr = [None] * world
            dist.all_gather_object(allr, mine)
        else:
            allr = [mine]
        res["per_rank"] = [{"rank": r[0], "max_iters": r[1], "mean_iters": r[2], "solve_ms": r[3], "gather_ms": r[4]} for r in allr]
        # residuals of the local shard, worst over ranks
        st = b.stage_stats()
        sst = last["stage_status"][:, solver.mine]
        worst = np.zeros((6, 3))
        for s in range(6):
            ran = sst[s] != -9
            if ran.any():
                worst[s] = st[s][ran][:, 1:4].max(axis=0)
        res["worst"] = reduce_max(worst.reshape(-1).tolist()).reshape(6, 3)
        if with_kernels:
            b.set_timing(True)
            b.kernel_times(reset=True)
            solver.solve(resident=True)
            res["kt"] = b.kernel_times(reset=True)
            b.set_timing(False)
            res["kt_iters"] = last["stage_iters"][:, solver.mine]
        return res

    sampler = ClockSampler(local)
    sampler.start()
    M = measure(per_gpu, args.steps, args.warmup, True)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    solver, problems = M["solver"], M["problems"]
    batch = solver.batch
    sz = batch.sizes.astype(np.int64)
    szf = batch.sizes_fixed().astype(np.int64)

    # e2e: public API with host buffers (layout build + H2D + solve + device sampling + gather + D2H), host clock
    # around fully synchronous calls; max over ranks
    def step_e2e():
        t0 = time.perf_counter()
        s2 = chd.parallel.ShardedSolver(problems, device=local, rank=rank, world=world)
        out = s2.solve()
        h2d = s2.batch.h2d_bytes()
        s2.close()
        return time.perf_counter() - t0, h2d, out["d2h_bytes"]
    step_e2e()
    barrier()
    e2e_t, h2d, d2h = [], 0, 0
    for _ in range(args.steps):
        dt, h2d, d2h = step_e2e()
        e2e_t.append(dt)
    barrier()
    e2e_total = float(reduce_max([sum(e2e_t)])[0])

    named = None
    if world == args.named_world and args.workload == "phys" and per_gpu != 128 and not args.no_named:
        # BASELINE.json configs[3]: 1024 sequences x 120 frames sharded across 8 B200 (128 per GPU)
        solver.close()
        Mn = measure(128, max(1, min(args.steps, 5)), 1, False)
        named = {"config": workload_config("phys", world, 128), "value": Mn["N"] * frames * max(1, min(args.steps, 5)) / Mn["t_total"],
                 "unit": "frames/s", "steps": max(1, min(args.steps, 5)), "warmup": 1, "ms_per_step": 1e3 * Mn["t_total"] / max(1, min(args.steps, 5)),
                 "per_rank": Mn["per_rank"],
                 "residual": residual_summary_gpu(np.zeros((6, Mn["N"], 4)), Mn["last"]["stage_status"], Mn["last"]["stage_iters"], Mn["last"]["success"]),
                 "note": "device-resident timing like `value`; the reference arm's value (frames/s of the fully loaded host) is the divisor for the >= 100x target"}
        for s in range(6):
            k = STAGE_NAMES[s]
            if k in named["residual"]:
                named["residual"][k]["max_nlp_error"], named["residual"][k]["max_constr_viol"], named["residual"][k]["max_dual_inf"] = \
                    [float(x) for x in Mn["worst"][s]]
        Mn["solver"].close()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak, peak_src = (peaks.get("hbm_gbs"), "measured") if peaks.get("hbm_gbs") else (6650.0, "fallback")
        last = M["last"]
        value = M["N"] * frames * args.steps / M["t_total"]
        kt = M["kt"]
        # dominant kernel: chd_k_kkt.  Algorithmic bytes per launch (DESIGN.md): per active sequence
        # 8*(nslots [J] + 2n [grad, dx] + 12m [row state in/out]); the band itself is scratch.  Every sequence walks
        # through the schedule at its own pace: units per launch = (sum of iterations over sequences and stages) / launches
        it = M["kt_iters"].astype(np.float64)                       # (6, B) of this rank
        seq_iters = it.sum(axis=0)
        kkt_ms, kkt_n = kt["kkt"]
        eval_ms, eval_n = kt["eval"]
        act = seq_iters / max(kkt_n, 1)
        launch_bytes = float((8 * (sz[:, 2] + 2 * sz[:, 0] + 12 * sz[:, 1]) * act).sum())
        ach = launch_bytes / (kkt_ms / max(kkt_n, 1) * 1e-3) / 1e9 if kkt_n else 0.0
        eval_bytes = float((8 * (2 * sz[:, 0] + 2 * sz[:, 1] + sz[:, 2] + (18 + 3 * n_ee) * frames) * act).sum())
        eval_ach = eval_bytes / (eval_ms / max(eval_n, 1) * 1e-3) / 1e9 if eval_n else 0.0
        traffic = None
        for fn in ("r2_kkt_ncu.json", "r1_kkt_ncu.json"):
            try:
                prof = json.load(open(os.path.join(ROOT, "profiles", fn)))
                traffic = prof["dram_bytes_per_sequence_per_launch"] * float(act.sum())   # ncu --set full capture, per launch
                break
            except Exception:
                pass
        # band LDL^T flops of one factorisation: Na * (w + nb + 1)^2 (Golub & Van Loan); stage 3 works with the wider
        # band / border (switch times), the other stages with (w_fix, nb_fix)
        def fl(w, nb):
            return sz[:, 3] * (w + nb + 1.0) ** 2
        it3 = it[4]
        kkt_flops = float(((seq_iters - it3) * fl(szf[:, 1], szf[:, 0]) + it3 * fl(sz[:, 5], sz[:, 4])).sum()) / max(kkt_n, 1)
        kkt_gflops = kkt_flops / (kkt_ms / max(kkt_n, 1) * 1e-3) / 1e9
        try:
            dfma_peak, dmma_peak = chd.phys.measure_fp64_peak()
        except Exception:
            dfma_peak = dmma_peak = None
        resid = residual_summary_gpu(np.zeros((6, M["N"], 4)), last["stage_status"], last["stage_iters"], last["success"])
        for s in range(6):
            k = STAGE_NAMES[s]
            if k in resid:
                resid[k]["max_nlp_error"], resid[k]["max_constr_viol"], resid[k]["max_dual_inf"] = [float(x) for x in M["worst"][s]]
        line = {
            "metric": "optimised frames/sec (batched phys-optim)", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * M["t_total"] / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.workload, world, per_gpu),
            "clocks": sampler.result(),
            "e2e": {"value": M["N"] * frames * args.steps / e2e_total, "unit": "frames/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "includes": "layout build, H2D, staged solve, device sampling, the NCCL gather (N>1), D2H"},
            "gpu_launches": int(M["launches"]),
            # dominant kernel: the KKT factorisation runs on the fp64 tensor-core pipe (DMMA) and is bound by that pipe's latency
            # chain, not by HBM (DESIGN.md section 3); its peak is measured in this run because MEASURED_PEAKS.json carries no
            # fp64 figure.  The HBM view of the same kernel (the north star asks for it) follows as `roofline_hbm`.
            "roofline": {"bound": "tensor", "kernel": "chd_k_kkt", "pipe": "fp64 tensor core (DMMA m8n8k4)",
                         "achieved": kkt_gflops / 1e3, "peak": (dmma_peak / 1e3) if dmma_peak else None, "unit": "TFLOP/s",
                         "frac": (kkt_gflops / dmma_peak) if dmma_peak else None, "traffic": traffic,
                         "peak_source": "chd_measure_fp64_peak: DMMA loop on all SMs, measured in this run (no fp64 entry in MEASURED_PEAKS.json)",
                         "peak_dfma": (dfma_peak / 1e3) if dfma_peak else None,
                         "algorithmic_flops": kkt_flops, "ms_per_launch": kkt_ms / max(kkt_n, 1),
                         "active_sequences_per_launch": float(act.sum()),
                         "note": "band LDL^T flop count Na*(w+nb+1)^2 per active sequence and factorisation; one CTA per sequence, so at "
                                 "most active_sequences_per_launch of the 148 SMs work"},
            "roofline_hbm": {"bound": "hbm", "kernel": "chd_k_kkt", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                             "frac": ach / hbm_peak, "traffic": traffic, "algorithmic_bytes": launch_bytes, "peak_source": peak_src},
            "kernels": {k: {"ms": v[0], "launches": v[1]} for k, v in kt.items()},
            "roofline_eval": {"bound": "hbm", "kernel": "chd_k_eval", "achieved": eval_ach, "peak": hbm_peak, "unit": "GB/s",
                              "frac": eval_ach / hbm_peak},
            "residual": resid,
            "per_rank": M["per_rank"],
        }
        if named:
            line["named_config_1024"] = named
        if not args.no_cpu and world == 1:
            cores = os.cpu_count() or 1
            fr_, ne_, de_ = frames, n_ee, dense
            seeds = list(range(min(cores, M["N"]))) if M["N"] >= cores else list(range(cores))
            v, wall, rc = cpu_arm(seeds, cores, fr_, ne_, de_)
            line["cpu_baseline"] = {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
                                    "sample": "%d sequences x %d frames (seeds 0..%d of the workload's generator), one per core on %d cores, "
                                              "full staged solve, %.1f s wall" % (len(seeds), fr_, len(seeds) - 1, cores, wall),
                                    "residual": rc}
        if args.dump_outputs:
            dump_outputs(last, args.dump_outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
