#!/usr/bin/env python
"""bench.py -- train-points/sec of the projected-process statistics hot path
(`getMatrixKmnKnmAndVectorKmny`, PGPH:20-36) on N B200s, next to the reference's CPU path.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py --gpus N --steps K --warmup W --dump-outputs DIR    (also writes DIR/G.npy, DIR/b.npy)

A "step" = one pass of the hot path over one batch of synthetic input: begin(active set) ->
accumulate(shard) -> finish (one ncclAllReduce of [G;b;status] across ranks).

Workloads (BASELINE.json `configs`; kernel `1*ARDRBFKernel(d) + 1.const*EyeKernel`, sigma2=1e-4, theta fixed at
C=1, beta_k=sqrt(18/d); X ~ U[0,1)^d generated in fp32, y = sin(sum x) + 0.1 eps):
  configs1 : synthetic 1M x 16 fp32 PER GPU, active=1000  (configs[1]; weak scaling)
  configs3 : synthetic 10M x 32 fp32 over 8 GPUs = 1.25M x 32 PER GPU, active=2000  (configs[3], the north-star target)
The PRIMARY line (`value`, `e2e`, `roofline`, `config`) is configs1 at N = 1, 2, 4 and configs3 at N = 8 -- the
configuration BASELINE.json quotes the 8-GPU target on; `series` carries BOTH workloads at every N (per-GPU shard
fixed = weak scaling in each series), so the 1 -> 8 efficiency of either series can be read from the per-N lines.

  value : inputs resident in HBM before the timed region (sgp_stats_accumulate_device), CUDA events on the
          library's stream, L2 flushed between steps (256 MiB memset).
  e2e   : the same step through the public host-buffer entry (sgp_stats_accumulate from pinned host
          memory, G and b copied back), host<->device copies inside the timed region.
  stats_plus_tail : value with the m x m tail (sgp_magic: K_mm, Cholesky PD check, magicVector, magicMatrix on rank 0's
          GPU) added to every step.
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (which may be read-only)

METRIC = "train_points_per_sec"
UNIT = "points/s"
N_E = 100
SIGMA2 = 1e-4
# the arithmetic the statistics kernel really computes in (the reference is fp64 throughout; north_star tolerance 1e-5)
DTYPE = "i8x3 digits (23-bit fixed point) -> exact i32 accumulate -> f64 fold; distances f16x2 split -> f32 (TMEM)"

WORKLOADS = {
    "configs1": dict(n_per_gpu=1_000_000, d=16, m=1000,
                     label="BASELINE configs[1]: synthetic 1M x 16 fp32 regression per GPU, active=1000"),
    "configs3": dict(n_per_gpu=1_250_000, d=32, m=2000,
                     label="BASELINE configs[3]: synthetic 10M x 32 fp32 regression over 8 GPUs (1.25M x 32 per GPU), "
                           "active=2000, one ncclAllReduce of the 2000 x 2000 + 2000 statistics"),
}


def primary_workload(n_gpus: int) -> str:
    return "configs3" if n_gpus == 8 else "configs1"


def workload_config(name: str, n_gpus: int) -> dict:
    w = WORKLOADS[name]
    return {"workload": "%s; expert=%d, 1*ARDRBFKernel(%d)+1.const*EyeKernel, sigma2=1e-4, C=1, beta=sqrt(18/d)"
                        % (w["label"], N_E, w["d"]),
            "name": name, "stage": "stats (K_mn + K_mn K_nm + K_mn y, all-reduced)", "n_per_gpu": w["n_per_gpu"],
            "d": w["d"], "m": w["m"], "n_total": w["n_per_gpu"] * n_gpus,
            "parallelism": "points sharded over %d GPU(s), one ncclAllReduce of [G;b]" % n_gpus,
            "l2": "flushed between timed steps (256 MiB memset)",
            "precision_mode": "SGP_PREC_AUTO -> tcgen05 int8 exact-accumulation kernel"}


def make_shard(name: str, rank: int):
    """X ~ U[0,1) generated in fp32 (the oracle consumes the same values up-cast), y = sin(sum x) + 0.1 eps."""
    w = WORKLOADS[name]
    rng = np.random.default_rng(13 + rank)
    X = rng.random((w["n_per_gpu"], w["d"]), dtype=np.float32)
    y = np.sin(X.astype(np.float64).sum(1)) + 0.1 * rng.standard_normal(w["n_per_gpu"])
    return X, y


def active_set(name: str):
    w = WORKLOADS[name]
    rng = np.random.default_rng(7)
    X0 = np.random.default_rng(13).random((w["n_per_gpu"], w["d"]), dtype=np.float32)
    return X0[rng.permutation(w["n_per_gpu"])[:w["m"]]].astype(np.float64)


def algorithmic_flops_per_point(m: int, d: int) -> float:
    """SURVEY 8(d): 2*m*d (distance contraction) + m*(m+1) (symmetric Gram) + 2*m (K_mn y)."""
    return 2.0 * m * d + m * (m + 1.0) + 2.0 * m


def cpu_sample_points(name: str, cores: int) -> int:
    """Bounded CPU sample (~10-30 s): per-expert work ~ m^2 n_e, so fewer experts per worker at m = 2000."""
    w = WORKLOADS[name]
    per_worker = 80 if w["m"] <= 1000 else 24
    return int(min(w["n_per_gpu"], max(cores * per_worker * N_E, 20_000)))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j.get("bf16_tflops_sustained", j["bf16_tflops"])), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1400.0, "fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)"


def ncu_traffic(name: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE Gram-kernel launch over this workload's per-GPU shard, from the
    newest committed `ncu --set full` summary (profiles/*_traffic.json written by tools/ncu_summary.py); None if the
    current kernel has no capture for this workload."""
    best, src = None, None
    for p in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json"))):
        try:
            j = json.load(open(p))
        except Exception:
            continue
        if j.get("workload") == name:
            best, src = j, os.path.basename(p)
    if best is None:
        return None, None
    return int(best["dram_bytes_per_launch"]), src


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.perf_counter()] + [c.strip() for c in line.split(",")])

    def stop(self, t_begin: float = 0.0, t_end: float = float("inf")) -> dict:
        """Median SM clock over the samples taken inside [t_begin, t_end] (host perf_counter), i.e. under load;
        throttle reasons over the same window.  The sampler runs from before the warm-up (20 ms period)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, all_sm = [], None, set(), []
        for row in self.rows:
            ts, r = row[0], row[1:]
            try:
                v_sm = float(r[0]); mx = float(r[1])
            except Exception:
                continue
            all_sm.append(v_sm)
            if ts < t_begin - 0.02 or ts > t_end + 0.02:
                continue
            sm.append(v_sm)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else (float(np.max(all_sm)) if all_sm else None), "sm_max_mhz": mx,
                "samples": len(sm), "samples_total": len(all_sm), "reasons": sorted(reasons)}


def oracle_factory(d: int):
    import oracle
    beta = np.full(d, np.sqrt(18.0 / d))
    return lambda: (1 * oracle.ARDRBFKernel(beta) + oracle.const(1) * oracle.EyeKernel()
                    + oracle.const(SIGMA2) * oracle.EyeKernel())


def time_cpu_port(name: str, steps: int, warmup: int):
    """The reference's CPU path (oracle port with the reference's structure, all usable host cores) on a bounded sample
    of workload `name`.  Returns (points/s, seconds per step, cores, sample points)."""
    from oracle.cpu_baseline import stats_parallel, usable_cores
    w = WORKLOADS[name]
    cores = usable_cores()
    sample = cpu_sample_points(name, cores)
    X, y = make_shard(name, 0)
    X, y = X[:sample].astype(np.float64), y[:sample]
    Z = active_set(name)
    fac = oracle_factory(w["d"])
    theta = fac().get_hyperparameters()
    for _ in range(warmup):
        stats_parallel(X[:4000], y[:4000], Z, fac, theta, N_E, cores)
    t = 0.0
    for _ in range(steps):
        _, _, dt = stats_parallel(X, y, Z, fac, theta, N_E, cores)
        t += dt
    return sample * steps / t, t / steps, cores, sample


# ------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CPU implementation of the path (here: the oracle port -- the reference is Scala
    and there is no JVM in this image), all host cores, on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = primary_workload(args.gpus)
    value, sec, cores, sample = time_cpu_port(name, args.steps, args.warmup)
    cpu = {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": "%d points of the %d-point shard per step (path is linear in N at fixed m,d,n_e)"
                     % (sample, WORKLOADS[name]["n_per_gpu"])}
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                      "data": "synthetic", "config": workload_config(name, args.gpus), "cpu_baseline": cpu,
                      "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0}))


def run_ours(args):
    import torch
    import torch.distributed as dist
    import spark_gp_b200 as sg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run)" % (args.gpus, world))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng = sg.ProjectedProcessEngine(local_rank)
    if world > 1:
        ids = [sg.ProjectedProcessEngine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        eng.comm_init(ids[0], rank, world)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def l2_flush():
        flush.zero_()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    prim = primary_workload(world)

    def measure(name: str, with_e2e: bool, steps: int, warmup: int, precision=None, keep_outputs=False):
        eng.set_precision(sg._native.SGP_PREC_AUTO if precision is None else precision)
        w = WORKLOADS[name]
        n, d, m = w["n_per_gpu"], w["d"], w["m"]
        Xh, yh = make_shard(name, rank)
        Z = active_set(name)
        beta = np.full(d, np.sqrt(18.0 / d))
        kernel = 1 * sg.ARDRBFKernel(beta) + sg.const(1) * sg.EyeKernel() + sg.const(SIGMA2) * sg.EyeKernel()
        Xd = torch.from_numpy(Xh).to(dev)
        yd = torch.from_numpy(yh).to(dev)

        def step_device():
            eng.event_record(0)
            eng.begin(kernel, Z)
            eng.accumulate_ptr(Xd.data_ptr(), True, yd.data_ptr(), n, device=True)
            eng.finish(copy_out=False)                    # all-reduce of [G;b]; statistics stay on the device
            eng.event_record(1)
            return eng.event_elapsed_ms(0, 1)

        for _ in range(warmup):
            step_device()
        path = eng.last_path()
        l2_flush()
        launches0 = eng.launch_count()
        barrier()
        t_wall0 = time.perf_counter()
        dev_ms, kern_ms, kern_n = 0.0, 0.0, 0
        for _ in range(steps):
            dev_ms += step_device()
            kms, kn = eng.gram_kernel_time()
            kern_ms += kms; kern_n += kn
            l2_flush()
            # every step ends in an all-reduce, so a rank that starts its step early spends the skew waiting INSIDE its
            # event-timed region: line the ranks up again (outside the timed region) before the next step
            barrier()
        t_wall1 = time.perf_counter()
        launches = eng.launch_count() - launches0
        res = {"name": name, "n": n, "d": d, "m": m, "dev_ms": dev_ms, "kern_ms": kern_ms, "kern_n": kern_n,
               "launches": launches, "t_wall": (t_wall0, t_wall1), "path": path, "e2e_ms": None}
        if keep_outputs:
            # the last timed step's all-reduced statistics, as a caller receives them: finishing a finished window
            # only copies the device-resident [G;b] out (no second all-reduce)
            res["outputs"] = dict(zip(("G", "b"), eng.finish()))

        # tail (m x m, fp64; rank 0 does it in a fit): statistics of the last step are still on the device
        eng.magic(copy_out=False)                       # first call pays cuSOLVER's lazy initialisation / workspace
        tails = []
        for _ in range(3):
            t0 = time.perf_counter()
            eng.magic(copy_out=False)
            tails.append(1e3 * (time.perf_counter() - t0))
        res["tail_ms"] = float(np.median(tails))

        if with_e2e:
            Xp = torch.from_numpy(Xh).pin_memory()
            yp = torch.from_numpy(yh).pin_memory()
            Gp = torch.empty((m, m), dtype=torch.float64).pin_memory()
            bp = torch.empty(m, dtype=torch.float64).pin_memory()

            def step_e2e():
                t0 = time.perf_counter()
                eng.begin(kernel, Z)
                eng.accumulate_ptr(Xp.data_ptr(), True, yp.data_ptr(), n, device=False)
                eng._check(eng._lib.sgp_stats_finish(eng._h, Gp.data_ptr(), bp.data_ptr()))
                return 1e3 * (time.perf_counter() - t0)

            for _ in range(max(1, min(warmup, 2))):
                step_e2e()
            barrier()
            e2e_ms = 0.0
            for _ in range(steps):
                e2e_ms += step_e2e()
                barrier()
            res["e2e_ms"] = e2e_ms
            res["h2d"] = int(n * d * 4 + n * 8 + m * d * 8)
            res["d2h"] = int((m * m + m) * 8)
            # multi-GPU correctness of the all-reduced statistics (outside every timed region): each rank recomputes
            # its LOCAL statistics with a second, communicator-less context and the ranks compare
            # sum_r trace(G_r), sum_r sum(b_r) with the all-reduced G, b every rank holds
            if world > 1:
                Gall, ball = Gp.numpy().copy(), bp.numpy().copy()
                e2 = sg.ProjectedProcessEngine(local_rank)
                e2.begin(kernel, Z)
                e2.accumulate_ptr(Xd.data_ptr(), True, yd.data_ptr(), n, device=True)
                Gl, bl = e2.finish()
                e2.close()
                loc = torch.tensor([np.trace(Gl), bl.sum(), np.abs(Gl).sum()], dtype=torch.float64, device=dev)
                dist.all_reduce(loc, op=dist.ReduceOp.SUM)
                glob_ = torch.tensor([np.trace(Gall), ball.sum(), np.abs(Gall).sum()], dtype=torch.float64, device=dev)
                gmax = glob_.clone()
                dist.all_reduce(gmax, op=dist.ReduceOp.MAX)
                gmin = glob_.clone()
                dist.all_reduce(gmin, op=dist.ReduceOp.MIN)
                loc, gmax, gmin = loc.cpu().numpy(), gmax.cpu().numpy(), gmin.cpu().numpy()
                res["allreduce_check"] = {
                    "trace_G_rel": float(abs(gmax[0] - loc[0]) / abs(loc[0])),
                    "sum_b_rel": float(abs(gmax[1] - loc[1]) / max(abs(loc[1]), 1e-300)),
                    "abs_G_rel": float(abs(gmax[2] - loc[2]) / abs(loc[2])),
                    "ranks_agree": bool(np.all(gmax == gmin)),
                    "what": "sum over ranks of each rank's local trace(G_r), sum(b_r), sum|G_r| (a second context "
                            "without communicator) vs the all-reduced statistics; ranks_agree = bit-identical on all ranks"}
            del Xp, yp
        del Xd, yd
        t = torch.tensor([res["dev_ms"], res["e2e_ms"] or 0.0, res["kern_ms"]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res["dev_ms"], e2e_max, res["kern_ms"] = [float(v) for v in t.tolist()]
        if with_e2e:
            res["e2e_ms"] = e2e_max
        return res

    def series_entry(r, steps):
        n_total = r["n"] * world
        ms = r["dev_ms"] / steps
        e = {"workload": WORKLOADS[r["name"]]["label"], "n_per_gpu": r["n"], "d": r["d"], "m": r["m"],
             "value": n_total / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "tail_ms": r["tail_ms"],
             "stats_plus_tail": n_total / ((ms + r["tail_ms"]) / 1e3),
             "kernel_path": {0: "f64", 1: "f64_strict", 2: "i8", 4: "i8_direct"}.get(r["path"], str(r["path"])),
             "gram_kernel_ms": r["kern_ms"] / max(r["kern_n"], 1)}
        if r["e2e_ms"]:
            e["e2e"] = n_total * steps / (r["e2e_ms"] / 1e3)
        return e

    other = "configs1" if prim == "configs3" else "configs3"
    rp = measure(prim, True, args.steps, args.warmup, keep_outputs=bool(args.dump_outputs) and rank == 0)
    if "outputs" in rp:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, v in rp.pop("outputs").items():
            np.save(os.path.join(args.dump_outputs, k + ".npy"), v)
    ro = measure(other, False, max(2, min(args.steps, 3)), 3)
    clocks = sampler.stop(*rp["t_wall"]) if rank == 0 else None
    rd = None
    if world == 1 and args.direct:      # same shard, exponents from direct fp32 distances (what AUTO picks for large norms)
        rd = measure("configs1", False, 3, 3, precision=sg._native.SGP_PREC_I8_DIRECT)
        eng.set_precision(sg._native.SGP_PREC_AUTO)

    if rank == 0:
        n_total = rp["n"] * world
        value = n_total * args.steps / (rp["dev_ms"] / 1e3)
        e2e_value = n_total * args.steps / (rp["e2e_ms"] / 1e3)
        peak_tf, peak_src = measured_peaks()
        launch_ms = rp["kern_ms"] / max(rp["kern_n"], 1)
        flops = algorithmic_flops_per_point(rp["m"], rp["d"]) * rp["n"] * args.steps / max(rp["kern_n"], 1)
        achieved_tf = flops / (launch_ms / 1e3) / 1e12
        traffic, traffic_src = ncu_traffic(prim)
        roof = {"bound": "tensor", "kernel": "kmn_gram_i8_ring_kernel", "achieved": achieved_tf, "peak": peak_tf,
                "unit": "TFLOP/s", "frac": achieved_tf / peak_tf, "peak_source": peak_src,
                "traffic": traffic, "traffic_source": traffic_src, "launch_ms": launch_ms,
                "launches_timed": rp["kern_n"], "algorithmic_flops_per_launch": flops,
                "note": "algorithmic flops = N*(2md + m(m+1) + 2m); the kernel executes 6 int8 products per Gram "
                        "tile pair (exact 23-bit arithmetic), none of the extra products is credited"}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            v, sec, cores, sample = time_cpu_port(prim, 1, 1)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": "%d points of the same shard, oracle restatement, %d worker processes" % (sample, cores)}
        ms_step = rp["dev_ms"] / args.steps
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
               "config": workload_config(prim, world), "clocks": clocks,
               "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": rp["e2e_ms"] / args.steps,
                       "h2d_bytes_per_step": rp["h2d"], "d2h_bytes_per_step": rp["d2h"]},
               "gpu_launches": int(rp["launches"]), "roofline": roof, "cpu_baseline": cpu,
               "tail_ms": rp["tail_ms"],
               "stats_plus_tail": {"value": n_total / ((ms_step + rp["tail_ms"]) / 1e3), "unit": UNIT,
                                   "ms_per_step": ms_step + rp["tail_ms"]},
               "series": {prim: series_entry(rp, args.steps), other: series_entry(ro, max(2, min(args.steps, 3)))},
               "wall_ms_timed_region": 1e3 * (rp["t_wall"][1] - rp["t_wall"][0])}
        if rd is not None:
            out["series"]["configs1_i8_direct"] = series_entry(rd, 3)
        if "allreduce_check" in rp:
            out["allreduce_check"] = rp["allreduce_check"]
        if world == 1 and args.fit:
            out["fit"] = fit_number(sg, args)
        if world == 1 and args.sweep:
            out["sweep"] = sweep_number(sg, eng, torch, dev)
        print(json.dumps(out))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def sweep_number(sg, eng, torch, dev):
    """BASELINE configs[4] shape per GPU (12.5M x 8, active=4000): the HBM-bound K_nm sweep -- materialise the fp32 cross
    kernel of a 262144-point chunk (the full shard's 200 GB of K_nm does not fit in HBM; the chunk buffer is rewritten),
    CUDA events on the library's stream, vs the measured HBM copy bandwidth."""
    n, d, m = 262_144, 8, 4000
    rng = np.random.default_rng(5)
    X = rng.random((n, d), dtype=np.float32)
    Z = X[rng.permutation(n)[:m]].astype(np.float64)
    kernel = 1 * sg.ARDRBFKernel(np.full(d, np.sqrt(18.0 / d))) + sg.const(1) * sg.EyeKernel()
    eng.begin(kernel, Z)
    Xd = torch.from_numpy(X).to(dev)
    Kd = torch.empty((n, m), dtype=torch.float32, device=dev)
    for _ in range(2):
        eng.kmn_sweep_device(Xd.data_ptr(), True, n, Kd.data_ptr())
    eng.sync()
    reps = 5
    eng.event_record(2)
    for _ in range(reps):
        eng.kmn_sweep_device(Xd.data_ptr(), True, n, Kd.data_ptr())
    eng.event_record(3)
    ms = eng.event_elapsed_ms(2, 3) / reps
    bytes_alg = n * m * 4.0 + n * d * 4.0
    peak = None
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    gbs = bytes_alg / (ms / 1e3) / 1e9
    return {"workload": "BASELINE configs[4] shard shape: K_nm sweep of %d x %d points against active=%d, fp32 out" % (n, d, m),
            "ms_per_chunk": ms, "points_per_sec": n / (ms / 1e3), "elements_per_sec": n * m / (ms / 1e3),
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": (gbs / peak) if peak else None,
                         "algorithmic_bytes": bytes_alg, "note": "bytes = n*m*4 written + n*d*4 read; prep of the fp16 images included"}}


def fit_number(sg, args):
    """SURVEY 8(d)(iv): whole GaussianProcessRegression.fit at a FIXED maxIter on the configs[1] shard
    (optimizeHypers on the per-expert BCM objective -> statistics -> tail), GaussianProcessCommons.scala:66-92, 40-59."""
    w = WORKLOADS["configs1"]
    X, y = make_shard("configs1", 0)
    d, m = w["d"], w["m"]
    max_iter = 10
    gp = (sg.GaussianProcessRegression().setKernel(lambda: 1 * sg.ARDRBFKernel(np.full(d, np.sqrt(18.0 / d)))
                                                   + sg.const(1) * sg.EyeKernel())
          .setDatasetSizeForExpert(N_E).setActiveSetSize(m).setSigma2(SIGMA2).setMaxIter(max_iter).setTol(1e-6).setSeed(13))
    gp.fit(X[:50_000], y[:50_000])                                      # warm-up: contexts, lazy library initialisation
    t0 = time.perf_counter()
    gp.fit(X, y)                                                        # first full-size fit: allocates every workspace
    dt_first = time.perf_counter() - t0
    dts = []
    for _ in range(3):                                                  # steady state (contexts and workspaces pooled)
        t0 = time.perf_counter()
        gp.fit(X, y)
        dts.append(time.perf_counter() - t0)
    dt = float(np.median(dts))
    info = gp.last_objective or {}
    return {"value": len(X) / dt, "unit": UNIT, "seconds": dt, "seconds_first_call": dt_first, "maxIter": max_iter,
            "objective_evaluations": info.get("evaluations"), "lbfgsb_iterations": info.get("iterations"),
            "what": "GaussianProcessRegression.fit(1M x 16, expert=100, active=1000): L-BFGS-B on the GPU BCM objective "
                    "(fixed maxIter) + projected-process statistics + tail, host wall clock; median of 3 after one full-size fit "
                    "(seconds_first_call = that first fit, which allocates the workspaces)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fit", dest="fit", action="store_false", help="skip the whole-fit number (N=1 only)")
    ap.add_argument("--no-sweep", dest="sweep", action="store_false", help="skip the K_nm sweep number (N=1 only)")
    ap.add_argument("--no-direct", dest="direct", action="store_false",
                    help="skip the direct-distance int8 series entry (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the statistics of the last timed step of the primary workload as DIR/G.npy (m x m) and "
                         "DIR/b.npy (m), float64: at most 32 MB (m = 2000); the inputs are seeded, so two builds can be "
                         "compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
