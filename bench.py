#!/usr/bin/env python
"""bench.py -- L-BFGS iterations/s (and apply_Hv HBM GB/s) on the BASELINE configs, default config 2:
paired Rosenbrock, n = 1e7, fp64, m = 10, More-Thuente line search, x0 = 0, on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4|c5] [--solver-loop resident|host]
                  [--dump-outputs DIR]
  (N > 1: launched under torchrun, one rank per GPU; c2/c3: n is sharded over the ranks ("strong" scaling);
   c5: --sharding problems (default; ranks take whole problems, no communication) or n (every problem split along n);
   c4: replicas only, N = 1)

K steps are timed.  --dump-outputs DIR (one GPU) writes what the last timed step returned as DIR/<name>.npy, float64: x (c2, c3:
downloaded after the timed region; c4 also grad and the trace of f), fx, gnorm, niter, nfev (c5: one entry per problem).  The inputs
are fixed by the config, so two builds can be compared output for output.

A "step" is one complete minimize() of the problem through the header-only C++ front on top of liblbfgs_b200.so (c2: 22 iterations /
50 objective evaluations).  `value` = iterations per second with the start point already resident in HBM; `e2e` = the same with the
start point coming from pinned host memory and the solution copied back every step.  For built-in objectives the front runs the
device-resident solve: ONE persistent kernel launch per minimize() (lbfgspp_b200/csrc/persist.cuh); `roofline` is for that kernel:
algorithmic bytes of its passes (accounted by the kernel itself, include/lbfgs_b200.h: lbfgs_b200_solver_profile) divided by its
duration measured with CUDA events around the launch on the launching stream.  `cpu_baseline` / `--impl reference` time the CPU
restatement of the reference (oracle/; the reference itself cannot be built: Eigen is absent) on this box's host cores.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    "c2": dict(n=10_000_000, m=10, ls="MoreThuente",
               workload="C2: paired Rosenbrock n=1e7 fp64, m=10, LineSearchMoreThuente, x0=0 (BASELINE.json configs[1])"),
    "c3": dict(n=1_000_000, m=20, ls="Bracketing", max_iterations=150,
               workload="C3: quadratic f = 1/2 x'Ax - b'x, A = diag(d) + 1/2 tridiag(-1,2,-1) (d = exp(U[0, ln 1e3]), seed 0), n=1e6 fp64, m=20, "
                        "LineSearchBracketing, x0=0; first 150 iterations (the reference's own run ends at iteration ~199 in its line-search "
                        "exception at the rounding floor of f, tests/golden/c3_full.json) (BASELINE.json configs[2])"),
    "c4": dict(n=1_000_000, m=6, ls="MoreThuente",
               workload="C4: paired Rosenbrock in the box [2,4]^n, n=1e6 fp64, LBFGSBSolver defaults (m=6), x0=3 (BASELINE.json configs[3])"),
    "c5": dict(n=1_000_000, m=10, ls="MoreThuente", B=64,
               workload="C5: B=64 independent paired Rosenbrock problems, n=1e6 fp64, m=10, LineSearchMoreThuente, x0_b ~ U[-1,1] seed 1000+b "
                        "(BASELINE.json configs[4])"),
}


def workload_config(name):
    c = CONFIGS[name]
    cfg = {"workload": c["workload"], "n": c["n"], "m": c["m"], "line_search": c["ls"], "x0": "zeros" if name in ("c2", "c3") else
           ("3.0" if name == "c4" else "U[-1,1], numpy default_rng(1000 + b)"), "params": "reference defaults except m"}
    if "max_iterations" in c:
        cfg["max_iterations"] = c["max_iterations"]
    if "B" in c:
        cfg["batch"] = c["B"]
    return cfg


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_SAMPLE = 1 << 21   # entries kept of a longer vector: 16 MB in float64, so a dump stays far below 64 MB


def dump_outputs(outdir, arrays):
    """Write each array as outdir/<name>.npy in float64.  A vector longer than DUMP_SAMPLE is replaced by its entries at DUMP_SAMPLE
    sorted indices drawn with seed 0 from its length: the same entries in every run."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.size > DUMP_SAMPLE:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(outdir, name + ".npy"), a)


def result_arrays(r, *extra):
    """What a caller of one minimize() receives, for --dump-outputs: the scalars and the named vectors of the result dict."""
    return {k: r[k] for k in ("fx", "gnorm", "niter", "nfev") + extra}


def load_traffic(key):
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as fh:
            return json.load(fh).get(key)
    return None


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md's clocks line).  Sampled in-process through NVML -- the
    library nvidia-smi itself reads -- every 50 ms: starting an nvidia-smi per sample re-initialises NVML every time and was seen to
    stall the solver's own driver calls (a 14 ms solve took 39 ms of wall clock on one box), and `nvidia-smi -lms` block-buffers its
    output into a pipe.  Falls back to one nvidia-smi process per sample when NVML cannot be loaded."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, gpu_index, gpu_uuid=None):
        super().__init__(daemon=True)
        self.idx = gpu_index
        self.uuid = gpu_uuid
        self.samples = []          # (sm_mhz, sm_max_mhz, set of active reasons)
        self.stop_flag = False
        self.source = None

    def _nvml_loop(self):
        import pynvml as nv
        nv.nvmlInit()
        h = None
        if self.uuid:
            for cand in (self.uuid, "GPU-" + self.uuid):
                try:
                    h = nv.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                    break
                except Exception:
                    try:
                        h = nv.nvmlDeviceGetHandleByUUID(cand)
                        break
                    except Exception:
                        h = None
        if h is None:
            h = nv.nvmlDeviceGetHandleByIndex(self.idx)
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        mx = int(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        self.source = "nvml"
        while not self.stop_flag:
            mask = int(get_reasons(h))
            self.samples.append((int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), mx, {k for k, b in bits.items() if mask & b}))
            time.sleep(0.05)
        try:
            nv.nvmlShutdown()
        except Exception:
            pass

    def _smi_loop(self):
        self.source = "nvidia-smi"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                f = [v.strip() for v in out.split(",")]
                if len(f) >= 7 and f[0].replace(".", "").isdigit():
                    self.samples.append((int(float(f[0])), int(float(f[1])), {k for k, v in zip(self.REASONS, f[3:7]) if v.lower().startswith("active")}))
            except Exception:
                pass
            time.sleep(0.1)

    def run(self):
        try:
            self._nvml_loop()
        except Exception:
            if not self.stop_flag:
                self._smi_loop()

    def summary(self):
        self.stop_flag = True
        self.join(timeout=8)
        sm = sorted(s[0] for s in self.samples)
        reasons = set()
        for s in self.samples:
            reasons |= s[2]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(s[1] for s in self.samples) if self.samples else None,
                "reasons": sorted(reasons), "samples": len(self.samples), "source": self.source}


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (oracle/ is executed only here, in tests/ and in smoke())
# ---------------------------------------------------------------------------------------------------------------------
def load_oracle():
    """The restatement's timing build (-O3 -march=native), compiled for the host it is timed on into a temporary directory (the
    tree may be read-only); the portable build of the tree when that compile fails."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle as po
    try:
        with tempfile.TemporaryDirectory(prefix="lbfgs_b200_bench_") as tmp:
            return po, po.Oracle("orc", path=po.build_native(tmp))   # loaded before the directory is removed
    except Exception:
        return po, po.Oracle("orc")


def cpu_solve(po, orc, name, sum_mode, problem=0, max_iterations=None):
    """One full minimize() of config `name` (problem b of the batch for c5) on the CPU checker.  Returns (result dict, seconds)."""
    import numpy as np
    c = CONFIGS[name]
    n, m = c["n"], c["m"]
    mi = c.get("max_iterations", 0) if max_iterations is None else max_iterations
    if name == "c4":
        prm = orc.default_param(lbfgsb=True, max_iterations=mi)
        r = orc.lbfgsb(po.OBJ_ROSENBROCK_PAIRED, np.full(n, 3.0), 2.0, 4.0, prm, sum_mode=sum_mode, trace_cap=4096)
    elif name == "c3":
        d, b, _ = po.quad_tridiag_data(n, kappa=1e3, seed=0)
        prm = orc.default_param(m=m, max_iterations=mi)
        r = orc.lbfgs(po.OBJ_QUAD_TRIDIAG, np.zeros(n), po.LS_BRACKETING, prm, data0=d, data1=b, sum_mode=sum_mode, trace_cap=4096)
    else:
        x0 = np.zeros(n) if name == "c2" else np.random.default_rng(1000 + problem).uniform(-1, 1, n)
        prm = orc.default_param(m=m, max_iterations=mi)
        r = orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, x0, po.LS_MORE_THUENTE, prm, sum_mode=sum_mode, trace_cap=4096)
    return r


def cpu_baseline_block(name, gpu_niter=None, gpu_nfev=None, gpu_fx=None):
    """The reported (not the target) CPU figure of the main arm: one full solve on ONE host thread -- the reference's Eigen level-1
    code is single-threaded and never enables OpenMP (SURVEY.md 8d)."""
    po, orc = load_oracle()
    r = cpu_solve(po, orc, name, po.SUM_LANES8)
    out = {"value": r["niter"] / r["seconds"], "unit": "iters/s", "cores": 1, "kind": "port",
           "sample": "1 x minimize() of the same problem%s (%d iterations, %d evaluations, %.1f s), single thread like the reference's Eigen "
                     "level-1 code, 8-lane partial sums; restatement of the reference (oracle/, -O3 -march=native)"
                     % (" (problem 0 of the batch)" if name == "c5" else "", r["niter"], r["nfev"], r["seconds"])}
    if gpu_niter is not None:
        out["niter_matches_gpu"] = bool(r["niter"] == gpu_niter and r["nfev"] == gpu_nfev)
        out["fx_abs_diff"] = abs(r["fx"] - gpu_fx)
    return out


def run_reference_arm(args, rank):
    """The reference's CPU implementation of the path on the host cores, pinned (VERDICT r1): the FULL solve of the config, ONE thread
    as `value` (the reference's own threading), the OpenMP restatement on all cores as an extra key; never truncated, never
    self-calibrated.  --steps is the number of timed solves (a solve of c2 takes ~12 s)."""
    if rank != 0:
        return
    name = args.config
    po, orc = load_oracle()
    cpu_solve(po, orc, name, po.SUM_LANES8, max_iterations=1)          # untimed: first touch of the allocator, library load
    nsolves = args.steps
    secs, iters, last = 0.0, 0, None
    for _ in range(nsolves):
        last = cpu_solve(po, orc, name, po.SUM_LANES8)
        secs += last["seconds"]
        iters += last["niter"]
    value = iters / secs
    allc = cpu_solve(po, orc, name, po.SUM_LANES8_OMP)
    all_cores = {"value": allc["niter"] / allc["seconds"], "unit": "iters/s", "cores": orc.hw_threads(),
                 "note": "the same full solve by the OpenMP build of the restatement on all host threads (the reference has no such mode)"}
    sample = ("%d x the full minimize() of the config (%d iterations, %d evaluations each), 1 thread; warm-up = one 1-iteration solve; "
              "restatement of the reference (oracle/, -O3 -march=native, 8-lane partial sums)" % (nsolves, last["niter"], last["nfev"]))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, result_arrays(last, "x"))
    ref_headers = None
    if name == "c2":
        try:   # for the record: the unmodified reference headers themselves (over the minieigen stand-in), 3 iterations of the same solve
            import numpy as np
            ref = po.Oracle("ref")
            rr = ref.lbfgs(po.OBJ_ROSENBROCK_PAIRED, np.zeros(CONFIGS[name]["n"]), po.LS_MORE_THUENTE,
                           ref.default_param(m=CONFIGS[name]["m"], max_iterations=3), trace_cap=64)
            ref_headers = {"value": rr["niter"] / rr["seconds"], "unit": "iters/s", "cores": 1,
                           "sample": "3 iterations of the same solve by oracle/_ref (reference headers compiled over oracle/minieigen, -O2)"}
        except Exception:  # noqa: BLE001  (no _ref build on this machine)
            pass
    line = {"impl": "reference", "metric": "lbfgs_iterations_per_sec", "value": value, "unit": "iters/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "timed_solves": nsolves, "ms_per_step": 1e3 * secs / nsolves, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(name),
            "cpu_baseline": {"value": value, "unit": "iters/s", "cores": 1, "kind": "port", "sample": sample, "all_cores": all_cores,
                             "reference_headers": ref_headers},
            "e2e": {"value": value, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--hv", default="auto", choices=["auto", "two_loop", "gram"], help="host-driven loop only")
    ap.add_argument("--comm", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: in-kernel exchange over NVLink peer memory (default; required by the device-resident solve) or one "
                         "ncclAllReduce per reduction (host-driven loop only)")
    ap.add_argument("--solver-loop", default="resident", choices=["resident", "host"],
                    help="device-resident solve (one persistent kernel launch per minimize; default) or the host-driven loop (one launch per pass)")
    ap.add_argument("--sharding", default="problems", choices=["problems", "n"], help="c5 on N > 1 GPUs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-mode", action="store_true", help="timed region only (for runs under ncu; numbers are not bench values)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float64; a vector longer than "
                         "%d entries as a fixed, seeded sample of that many)" % DUMP_SAMPLE)
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    return args


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        sys.exit("--dump-outputs runs on one GPU")

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import numpy as np
    import torch
    import lbfgspp_b200 as lb

    assert torch.cuda.is_available(), "bench.py needs a B200 (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t)
        return float(t.item())

    name = args.config
    cfg = CONFIGS[name]
    n_global, m_hist = cfg["n"], cfg["m"]
    from lbfgspp_b200.sharding import shard_bounds
    shard_n = world > 1 and (name in ("c2", "c3") or (name == "c5" and args.sharding == "n"))
    assert not (name == "c4" and world > 1), "config 4 (L-BFGS-B) runs as replicas only: use --gpus 1"
    lo, hi = shard_bounds(n_global, rank, world) if shard_n else (0, n_global)
    n_local = hi - lo
    resident = args.solver_loop == "resident" and name != "c4"
    if shard_n and args.comm == "nccl":
        assert not resident, "--comm nccl needs --solver-loop host"
        ident = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            ident = torch.tensor(list(lb.comm_unique_id()), dtype=torch.uint8, device="cuda")
        dist.broadcast(ident, src=0)
        lb.comm_init(local_rank, bytes(ident.cpu().numpy().tobytes()), rank, world, index_offset=lo)
    elif shard_n:
        mine = torch.tensor(list(lb.p2p_export(local_rank)), dtype=torch.uint8, device="cuda")
        allh = [torch.zeros(64, dtype=torch.uint8, device="cuda") for _ in range(world)]
        dist.all_gather(allh, mine)
        lb.p2p_attach(local_rank, b"".join(bytes(t.cpu().numpy().tobytes()) for t in allh), rank, world, index_offset=lo)
        if name == "c3":
            lb.set_global_extent(local_rank, lo, n_global)

    ctx = lb.driver_ctx(local_rank)
    abi = lb.abi()
    peak, peak_src = load_peaks()
    try:
        gpu_uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        gpu_uuid = None
    sampler = ClockSampler(local_rank, gpu_uuid)

    line = {"metric": "lbfgs_iterations_per_sec", "unit": "iters/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(name)}
    outputs = None   # --dump-outputs: name -> array of the last timed step

    def device_timed(fn, steps):
        """fn() `steps` times between a barrier + synchronize on both sides; CUDA-event time on the library's stream, max over ranks."""
        barrier()
        abi.lbfgs_b200_timer_start(ctx)
        outs = [fn() for _ in range(steps)]
        ms = C.c_float(0)
        abi.lbfgs_b200_timer_stop(ctx, C.byref(ms))
        barrier()
        return outs, max_over_ranks(ms.value * 1e-3)

    def roofline_from_profiles(profs, kernel_name, traffic_key):
        """profs: Session.profile() of every timed solve.  achieved = algorithmic bytes of the launch / its CUDA-event duration."""
        nbytes = sum(sum(v["alg_bytes"] for v in p["ops"].values()) for p in profs)
        ms = sum(p["kernel_ms"] for p in profs)
        ops = {}
        for p in profs:
            for k, v in p["ops"].items():
                o = ops.setdefault(k, dict(ms=0.0, rounds=0, alg_bytes=0.0))
                o["ms"] += v["ms"]; o["rounds"] += v["rounds"]; o["alg_bytes"] += v["alg_bytes"]
        ach = nbytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        return {"kernel": kernel_name, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": load_traffic(traffic_key), "peak_source": peak_src,
                "algorithmic_bytes": "per launch (= one minimize): sum over the kernel's passes of whole vectors read + written, 8 n x "
                                     "{first 3, trial 4, pair-forming dots 2c+4, combination + first trial 2c+3 (+2 when its x, g are stored), plain dots 2c+1, "
                                     "materialise 4}, c = pairs taking part in that pass; one iteration with T trials moves (4c+9) + 4(T-1) words per "
                                     "coordinate where SURVEY.md 8d counts (4c+2) + 6 + 8T for the unfused sequence",
                "launches_timed": len(profs), "ms_per_launch": ms / max(1, len(profs)),
                "passes": {k: {"ms_per_solve": v["ms"] / len(profs), "rounds_per_solve": v["rounds"] / len(profs),
                               "gb_per_s": v["alg_bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] > 0 else None} for k, v in ops.items()},
                "sync_ms_per_solve": sum(p["sync_ms"] for p in profs) / len(profs),
                "sync_wait_last_cta_ms_per_solve": sum(p["wait_last_cta_ms"] for p in profs) / len(profs),
                "sync_cross_rank_exchange_ms_per_solve": sum(p["exchange_ms"] for p in profs) / len(profs)}

    # ================================================================================================================ c2 / c3
    if name in ("c2", "c3"):
        if name == "c2":
            objective, data0, data1, x0 = lb.OBJ_ROSENBROCK_PAIRED, None, None, np.zeros(n_local)
            prm = lb.LBFGSParam(m=m_hist)
        else:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import pyoracle as po     # only the deterministic problem data generator (numpy), no CPU solver on the GPU arm
            d, b, _ = po.quad_tridiag_data(n_global, kappa=1e3, seed=0)
            objective, data0, data1, x0 = lb.OBJ_QUAD_TRIDIAG, d[lo:hi], b[lo:hi], np.zeros(n_local)
            prm = lb.LBFGSParam(m=m_hist, max_iterations=cfg["max_iterations"])
        hv = {"auto": lb.HV_AUTO, "two_loop": lb.HV_TWO_LOOP, "gram": lb.HV_GRAM}[args.hv]
        sess = lb.Session(objective, x0, prm, cfg["ls"], device=local_rank, hv_algo=hv, data0=data0, data1=data1, resident=resident)
        for _ in range(args.warmup):
            r = sess.solve()
        niter, nfev = r["niter"], r["nfev"]
        sampler.start()
        profs = []

        def one():
            rr = sess.solve()
            if resident:
                profs.append(sess.profile())
            return rr
        outs, dev_seconds = device_timed(one, args.steps)
        if args.dump_outputs:   # before the end-to-end solves below overwrite x
            outputs = dict(result_arrays(outs[-1]), x=sess.download())
        iters = sum(o["niter"] for o in outs)
        launches = sum(o["launches"] for o in outs)
        # ---- end to end: pinned host -> device every step, result back to the host ----
        for _ in range(0 if args.profile_mode else 2):
            sess.solve(from_host=True, to_host=True)
        barrier()
        t0 = time.perf_counter()
        e2e_iters, h2d, d2h = 0, 0, 0
        for _ in range(1 if args.profile_mode else args.steps):
            r2 = sess.solve(from_host=True, to_host=True)
            e2e_iters += r2["niter"]
            h2d, d2h = r2["h2d_bytes"], r2["d2h_bytes"] + 8  # + the fx scalar
        barrier()
        e2e_seconds = max_over_ranks(time.perf_counter() - t0)
        clocks = sampler.summary()
        line.update({"value": iters / dev_seconds, "ms_per_step": 1e3 * dev_seconds / args.steps, "scaling": "strong", "clocks": clocks,
                     "e2e": {"value": e2e_iters / e2e_seconds, "unit": "iters/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                     "gpu_launches": int(launches), "launches_per_solve": launches / args.steps,
                     "solver_loop": "device-resident: one persistent cooperative kernel launch per minimize()" if resident else "host-driven (one launch per pass)"})
        line["setup"] = {"n_per_gpu": n_local, "step": "one full minimize(): %d iterations, %d objective evaluations" % (niter, nfev),
                         "sharding": "single GPU, no collective" if world == 1 else
                         "n split over %d ranks; one exchange of the partial sums per pass %s" % (
                             world, "inside the kernel over NVLink peer memory" if args.comm == "p2p" else "with ncclAllReduce"),
                         "l2": "inputs larger than L2 (S,Y = %.2f GB per GPU)" % (2 * 8 * n_local * (m_hist + 1) / 1e9)}
        if resident:
            line["roofline"] = roofline_from_profiles(profs, "k_persist (device-resident solve)", "k_persist_dram_bytes_per_launch_%s" % name)
        # ---- the other loop, for comparison (not the headline) ----
        if not args.profile_mode and world == 1:
            other = lb.Session(objective, x0, prm, cfg["ls"], device=local_rank, hv_algo=hv, data0=data0, data1=data1, resident=not resident)
            for _ in range(3):
                other.solve()
            o_outs, o_secs = device_timed(other.solve, max(3, args.steps // 2))
            line["other_loop"] = {"solver_loop": "host-driven" if resident else "device-resident",
                                  "value": sum(o["niter"] for o in o_outs) / o_secs, "unit": "iters/s",
                                  "launches_per_solve": sum(o["launches"] for o in o_outs) / len(o_outs)}
            other.close()
        # ---- apply_Hv alone on a full history (c = m): the second half of BASELINE's metric ----
        if world == 1 and not args.profile_mode:
            rng = np.random.default_rng(0)
            mctx = lb.Context(local_rank)
            hist = lb.History(mctx, n_local, m_hist)
            blk = rng.standard_normal(1 << 20)

            def noise(seed):
                return np.resize(np.roll(blk, seed * 7919), n_local)
            for k in range(m_hist):
                s = noise(k)
                hist.add(mctx.array(s), mctx.array(s + 0.1 * noise(100 + k)))
            v, res = mctx.array(noise(999)), mctx.empty(n_local)
            for _ in range(3):
                hist.apply_Hv(v, -1.0, res, lb.HV_AUTO)
            reps = 30
            mctx.timer_start()
            for _ in range(reps):
                hist.apply_Hv(v, -1.0, res, lb.HV_AUTO)
            hv_ms = mctx.timer_stop() / reps
            gbs = 8.0 * n_local * (4 * m_hist + 2) / hv_ms / 1e6
            line["apply_Hv"] = {"ms_per_call": hv_ms, "gb_per_s": gbs, "frac_of_peak": gbs / peak, "c": m_hist,
                                "algorithmic_bytes": "8*n*(4c+2) per lbfgs_b200_hist_apply_Hv call (k_gram_dots + k_gram_combine), SURVEY.md 8d"}
        if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.profile_mode:
            line["cpu_baseline"] = cpu_baseline_block(name, niter, nfev, r["fx"])
        sess.close()

    # ================================================================================================================ c4
    elif name == "c4":
        solver = lb.LBFGSBSolver(lb.LBFGSBParam())
        x0 = np.full(n_global, 3.0)
        for _ in range(args.warmup):
            r = solver.minimize(lb.OBJ_ROSENBROCK_PAIRED, x0, 2.0, 4.0, trace_cap=256)
        sampler.start()
        barrier()
        secs, e2e_secs, iters, launches = 0.0, 0.0, 0, 0
        for _ in range(args.steps):
            r = solver.minimize(lb.OBJ_ROSENBROCK_PAIRED, x0, 2.0, 4.0, trace_cap=256)
            secs += r["seconds"]; e2e_secs += r["seconds_e2e"]; iters += r["niter"]; launches += r["launches"]
        barrier()
        clocks = sampler.summary()
        outputs = result_arrays(r, "x", "grad", "trace")
        # algorithmic bytes of one L-BFGS-B iteration at c pairs (DESIGN.md section 9): line-search trials 4n each, breakpoints + classes 5n,
        # W'd and the Cauchy build ~(2c+4)n, subspace minimisation >= (4c+8)n per BOXCQP sweep: reported as a lower bound with T trials
        nfev = r["nfev"]
        alg = 8.0 * n_global * (4.0 * nfev + r["niter"] * (5.0 + 2 * m_hist + 4 + 4 * m_hist + 8))
        ach = alg / (secs / args.steps) / 1e9
        line.update({"value": iters / secs, "ms_per_step": 1e3 * secs / args.steps, "scaling": "replicas only", "clocks": clocks,
                     "e2e": {"value": iters / e2e_secs, "unit": "iters/s", "h2d_bytes_per_step": 3 * 8 * n_global, "d2h_bytes_per_step": 2 * 8 * n_global + 8},
                     "gpu_launches": int(launches), "launches_per_solve": launches / args.steps,
                     "solver_loop": "host-driven (LBFGSBSolver: Cauchy point, subspace minimisation and More-Thuente trials as separate launches)",
                     "timing": "host wall clock around the synchronised minimize() (the L-BFGS-B loop interleaves host algebra on 2m x 2m matrices)",
                     "setup": {"step": "one full minimize(): %d iterations, %d objective evaluations" % (r["niter"], nfev)},
                     "roofline": {"kernel": "whole LBFGSBSolver iteration (many short launches)", "bound": "hbm", "achieved": ach, "peak": peak,
                                  "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                                  "algorithmic_bytes": "lower bound 8n[4 nfev + niter((2c+9) + (4c+8))] (trials; breakpoints/classes/Cauchy build; one "
                                                       "BOXCQP sweep), c = m = 6: the path is launch- and host-latency-bound at n = 1e6, not HBM-bound"}})
        # per-phase wall clock of the host-driven loop (LBFGSpp/PhaseClock.h: every scope synchronises, so the sum exceeds the untimed run)
        lb.phase_clock(True)
        for _ in range(2):
            solver.minimize(lb.OBJ_ROSENBROCK_PAIRED, x0, 2.0, 4.0, trace_cap=256)
        rep = lb.phase_report()
        lb.phase_clock(False)
        line["phases_ms_per_solve"] = {k: {"ms": 1e3 * v["seconds"] / 2, "calls": v["calls"] / 2} for k, v in rep.items()}
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_block(name, r["niter"], r["nfev"], r["fx"])

    # ================================================================================================================ c5
    else:
        B = cfg["B"]
        if shard_n:
            mine = list(range(B))
            X0 = np.stack([np.random.default_rng(1000 + b).uniform(-1, 1, n_global)[lo:hi] for b in mine])
        else:
            mine = list(range(rank, B, world))
            X0 = np.stack([np.random.default_rng(1000 + b).uniform(-1, 1, n_global) for b in mine])
        prm = lb.LBFGSParam(m=m_hist)
        bs = lb.BatchSession(lb.OBJ_ROSENBROCK_PAIRED, X0, prm, cfg["ls"], device=local_rank)
        for _ in range(max(1, min(args.warmup, 2))):
            res, _, _ = bs.solve(return_x=False)
        sampler.start()
        profs = []

        def one_batch():
            rr = bs.solve(return_x=False)[0]
            pr = bs.profile()
            if pr:
                profs.append(pr)
            return rr
        outs, dev_seconds = device_timed(one_batch, args.steps)
        iters_rank = sum(sum(p["niter"] for p in o) for o in outs)
        iters = iters_rank if shard_n else sum_over_ranks(iters_rank)
        barrier()
        t0 = time.perf_counter()
        h2d_bytes = bs.upload(X0)                 # end to end: the start points come from host memory ...
        resx, X, _ = bs.solve(return_x=True)      # ... and the solutions go back to it
        barrier()
        e2e_seconds = max_over_ranks(time.perf_counter() - t0)
        e2e_iters = sum(p["niter"] for p in resx) if shard_n else sum_over_ranks(sum(p["niter"] for p in resx))
        clocks = sampler.summary()
        outputs = {k: [p[k] for p in outs[-1]] for k in ("fx", "gnorm", "niter", "nfev")}
        its = [p["niter"] for p in outs[-1]]
        rounds = [p["rounds"] for p in outs[-1]]
        line.update({"value": iters / dev_seconds, "ms_per_step": 1e3 * dev_seconds / args.steps, "scaling": "strong", "clocks": clocks,
                     "e2e": {"value": e2e_iters / e2e_seconds, "unit": "iters/s", "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(X.nbytes),
                             "note": "one batched solve with its start points uploaded from and its solutions copied back to host memory (bytes per rank)"},
                     "gpu_launches": args.steps, "launches_per_solve": 1,
                     "solver_loop": "device-resident: ONE persistent kernel launch for the rank's whole batch",
                     "setup": {"problems_per_rank": len(mine), "n_per_gpu": n_local,
                               "sharding": "single GPU" if world == 1 else ("n of every problem split over %d ranks: one exchange per round carrying the "
                                                                            "partial sums of all running problems" % world if shard_n else
                                                                            "problem-parallel: rank r solves problems r, r+N, ...; no communication"),
                               "step": "one batched minimize(): %d problems, iterations min/mean/max = %d/%.0f/%d, rounds (streaming passes) of the longest = %d"
                                       % (len(its), min(its), float(np.mean(its)), max(its), max(rounds)),
                               "converged": int(sum(p["status"] == "ok" for p in outs[-1]))}})
        if profs:
            line["roofline"] = roofline_from_profiles(profs, "k_persist (device-resident solve, %d problems in one launch)" % len(mine), "k_persist_dram_bytes_per_launch_c5")
        if not args.no_cpu_baseline and rank == 0 and world == 1:
            line["cpu_baseline"] = cpu_baseline_block(name)
        bs.close()

    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
