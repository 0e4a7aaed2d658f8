#!/usr/bin/env python
"""bench.py -- the MCMC step path on BASELINE.json's configs, one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W]            (torchrun launches N > 1)
    python bench.py --impl reference ...                            CPU arm: the unmodified reference
    python bench.py ... --dump-outputs DIR                          also write the last timed step's outputs
                                                                    as DIR/<name>.npy (dumpOutputs)

N = 1  workload = config 3 ("synthetic hierarchical linear regression, partial pooling: 1,024 groups x
       200 obs x 8 coefficients, 1,024 chains x 20k iterations on 1 B200").
         value      chain-iterations/s over K timed steps of --iters-per-step iterations each, inputs resident
                    in HBM, on a slice of the config's schedule (burn-in with tuning, then thinning);
         e2e        the WHOLE config through the reference's own call: samplePosterior(1,024 chains, 20,000
                    iterations, nSamples 1,000) with the observations in host numpy arrays and the retained rows
                    streamed to sample/samples.npy -- chains x iterations / wall time of the call -- then
                    sampleDiagnosis.Diagnostic on those files: R-hat, min ESS, min ESS/s (`full_run`);
         also       16,384 chains on one GPU (config 4's single-GPU point) and config 5 (Bernoulli-logit,
                    partial and no pooling) as sub-records; the unmodified reference timed on the host cores.
N > 1  workload = config 4: the same model, 16,384 chains in total, 16,384 / N per GPU ("scaling": "strong");
       the between-chain diagnostics of the retained rows -- NCCL all-gather of half-chain summaries and the
       key-partitioned all-to-all behind the pooled median / HDI -- are timed and reported (`diagnostics`).

One step = ITERS_PER_STEP sampler iterations (posteriorSampling.py:862-896: P sweeps, P Gibbs hyper-updates,
tuning while burning in, retained-sample write-back after) of every chain.
"""

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "mcmc-for-nested-data_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from workloads import makeWorkload, makeLogitWorkload  # noqa: E402

METRIC = "chain-iterations/sec"
UNIT = "chain-iterations/s"
FLOP_PER_EVAL = 20.0      # 2K+4 at K=8 (SURVEY.md section 8d; DESIGN.md "algorithmic work"); 2K+4 for other K
C4_CHAINS = 16384
DUMP_BYTES = 60 * 10 ** 6     # --dump-outputs writes at most this much array data in all
REF_RUNNER = os.path.join(ROOT, "baseline", "run_reference.py")
REF_STAGED = os.path.join(ROOT, "baseline", "_ref", "posteriorSampling.py")
# DRAM bytes per step-kernel launch from the committed `ncu --set full` captures (dram__bytes_read.sum +
# dram__bytes_write.sum); they cannot be measured outside a profiler, so the capture is named beside the number
TRAFFIC = {"tc": (199.8e6, "profiles/r2_tc_kernel_ncu_summary.txt (1,024 chains: 180.2 MB read + 19.6 MB written)"),
           "pipe": (204.2e6, "profiles/r1_sweep_kernel_ncu_summary.txt (1,024 chains)"),
           "c5": (2.499e9, "profiles/r2_c5_kernel_ncu_summary.txt (4,096 chains: 1.673 GB read + 0.826 GB written)")}


def fixedPriors(pooling, coef):
    """Priors of the no-pooling variant (SURVEY.md section 8d: C5 uses N(0, 5) x 2; the regression
    shape N(0, 10) on the coefficients and Gamma(2) on sigma); None for partial pooling."""
    if pooling == "partial":
        return None
    import scipy.stats
    if coef == 0:
        return [scipy.stats.norm(0, 5), scipy.stats.norm(0, 5)]
    return [scipy.stats.norm(0, 10)] * coef + [scipy.stats.gamma(2)]


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(numpy.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- CPU arms
def _cpuChainWorker(job):
    """One chain of the oracle port for `nIter` iterations at the bench shape; returns the seconds
    spent in the iteration loop (data generation and start-up excluded, like the GPU arm)."""
    chain, nIter, G, R, K, pooling = job
    from oracle import posterior_oracle as po
    if K == 0:                                   # C5: Bernoulli-logit
        x, y, names, ranges = makeLogitWorkload(G, R)
        obj = po.BernoulliLogitObjective(x, y)
    else:
        X, y, names, ranges = makeWorkload(G, R, K)
        obj = po.LinearRegressionObjective(X, y)
    oc = po.OracleChain(chain, chain, max(nIter, 10), max(nIter, 10) // 2, names, G, R, pooling,
                        obj, fixedPriors(pooling, K), False, ranges)
    oc.nIter = nIter
    t0 = time.perf_counter()
    oc.run(keepRows=False)
    return time.perf_counter() - t0


def portBaseline(args, cores, iters):
    """chain-iterations/s of the oracle port (the reference's algorithm restated in numpy) on `cores` host
    processes, `iters` iterations of one chain each; the rate is over the slowest worker's loop time."""
    import multiprocessing
    jobs = [(c, iters, args.groups, args.obs, args.coef, args.pooling) for c in range(cores)]
    if cores == 1:
        loops = [_cpuChainWorker(jobs[0])]
    else:
        with multiprocessing.get_context("fork").Pool(cores) as pool:
            loops = pool.map(_cpuChainWorker, jobs)
    dt = max(loops)
    return cores * iters / dt, dt


def referenceRun(args, groups, chains, processes, iters):
    """One samplePosterior call of the UNMODIFIED reference (baseline/run_reference.py, own process) on
    the first `groups` groups of the workload.  Returns its JSON record."""
    cmd = [sys.executable, REF_RUNNER, "--groups", str(groups), "--obs", str(args.obs), "--coef", str(args.coef),
           "--pooling", args.pooling, "--chains", str(chains), "--processes", str(processes), "--iters", str(iters),
           "--full-groups", str(args.groups)]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=tempfile.gettempdir())
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        raise RuntimeError("reference run failed: " + r.stderr[-2000:])
    return json.loads(lines[-1])


def referenceRate(args, rec):
    """chain-iterations/s AT THE FULL SHAPE from a run on a slice of the groups: the reference's time per
    iteration is linear in the number of groups (Python loops over groups and observations,
    posteriorSampling.py:599-635; checked by the calibration run), so the rate scales by groups / full groups."""
    loop = max(rec["loop_s"])
    return rec["chains"] * rec["iters"] / loop * (float(rec["groups"]) / args.groups), loop


def referenceSampleText(args, rec):
    return ("unmodified reference (baseline/_ref, samplePosterior with a numpy objective in the style of "
            "example/regression.py), %d chain(s) on %d process(es) x %d iterations on the first %d of the %d groups "
            "(all %d observations x %d parameters of each), iteration loop only (from the reference's own log "
            "lines), rate scaled by %d/%d to the full shape"
            % (rec["chains"], rec["processes"], rec["iters"], rec["groups"], args.groups, args.obs,
               (args.coef + 1) if args.coef else 2, rec["groups"], args.groups))


def cpuBaselineRecord(args):
    """`cpu_baseline` of the GPU arm: the unmodified reference, one process, a bounded sample (about 10-20 s of
    CPU work); the oracle port beside it.  Falls back to the port alone when baseline/_ref is not staged."""
    out = {}
    v, dt = portBaseline(args, 1, args.cpu_iters)
    port = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "1 chain x %d iterations of the same workload at full shape (%.1f s in the loop), numpy "
                      "restatement of the reference (oracle/)" % (args.cpu_iters, dt)}
    if os.path.exists(REF_STAGED):
        rec = referenceRun(args, args.ref_groups, 1, 1, args.ref_iters * 2)
        rate, loop = referenceRate(args, rec)
        out = {"value": rate, "unit": UNIT, "cores": 1, "kind": "reference",
               "sample": referenceSampleText(args, rec) + " (%.1f s in the loop)" % loop,
               "numpy": rec["numpy"], "scipy": rec["scipy"], "port": port}
    else:
        out = port
    return out


def runReference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    world = int(os.environ.get("WORLD_SIZE", "1"))
    chainsCfg = args.chains_per_gpu if world == 1 else C4_CHAINS // world
    P, N = (args.coef + 1 if args.coef else 2), args.groups * args.obs
    staged = os.path.exists(REF_STAGED) and not args.port
    extra = {}
    if staged:
        for _ in range(args.warmup):
            referenceRun(args, args.ref_groups, cores, cores, args.ref_iters)
        t0 = time.perf_counter()
        rates, loops = [], []
        for _ in range(args.steps):
            rec = referenceRun(args, args.ref_groups, cores, cores, args.ref_iters)
            rate, loop = referenceRate(args, rec)
            rates.append(rate)
            loops.append(loop)
        dt = time.perf_counter() - t0
        value = cores * args.ref_iters * args.steps / sum(loops) * (float(args.ref_groups) / args.groups)
        kind, sample = "reference", referenceSampleText(args, rec) + "; per step"
        # calibration at the FULL shape, once: one process, and one process per core
        if not args.no_calibration:
            one = referenceRun(args, args.groups, 1, 1, args.ref_calibration_iters)
            allc = referenceRun(args, args.groups, cores, cores, args.ref_calibration_iters)
            extra = {"full_shape_1_process": {"value": one["chains"] * one["iters"] / max(one["loop_s"]), "unit": UNIT,
                                              "loop_s": max(one["loop_s"]), "wall_s": one["wall_s"]},
                     "full_shape_1_process_per_core": {"value": allc["chains"] * allc["iters"] / max(allc["loop_s"]),
                                                       "unit": UNIT, "cores": cores, "loop_s": max(allc["loop_s"]),
                                                       "wall_s": allc["wall_s"]},
                     "iterations": args.ref_calibration_iters, "numpy": one["numpy"], "scipy": one["scipy"],
                     "note": "the unmodified reference on ALL %d groups: the figure the scaled per-step rate must "
                             "reproduce" % args.groups}
    else:
        for _ in range(args.warmup):
            portBaseline(args, cores, 1)
        t0 = time.perf_counter()
        loops = []
        for _ in range(args.steps):
            loops.append(portBaseline(args, cores, args.port_iters)[1])
        dt = time.perf_counter() - t0
        value = cores * args.port_iters * args.steps / sum(loops)
        kind = "port"
        sample = ("%d chains (one per host core) x %d iterations per step of the same workload at full shape, numpy "
                  "restatement of the reference (oracle/), iteration loop only" % (cores, args.port_iters))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak" if world == 1 else "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workloadConfig(args, chainsCfg, world),
            "evals_per_sec": value * P * N,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if extra:
        line["cpu_baseline_reference"] = extra
    emit(json.dumps(line))


def workloadConfig(args, chains, world=1):
    pool = {"partial": "partial pooling", "none": "no pooling (fixed priors)"}[args.pooling]
    if not args.coef:
        name = "C5: hierarchical Bernoulli-logit, %s, %d groups x %d trials, 2 parameters" % (pool, args.groups, args.obs)
    elif world > 1:
        name = ("C4: hierarchical linear regression, %s, %d groups x %d obs x %d coefficients (+sigma), %d chains "
                "sharded over %d GPUs" % (pool, args.groups, args.obs, args.coef, chains * world, world))
    else:
        name = ("C3: hierarchical linear regression, %s, %d groups x %d obs x %d coefficients (+sigma)"
                % (pool, args.groups, args.obs, args.coef))
    return {"workload": name,
            "chains_per_gpu": chains, "iters_per_step": args.iters_per_step,
            "schedule": "burn = first half of the run (tune every 100), thin %d after" % args.thin,
            "l2": "chain state + sample write-back exceed L2 (%.0f MB touched per iteration)"
                  % (chains * args.groups * ((args.coef + 1) if args.coef else 2) * 28 / 1e6)}


def roofline(args, tensorCore, sweepMs, chains, peakFp32, peakTf32, peakMufu):
    """Roofline of the step kernel (DESIGN.md section 4).  Algorithmic work per chain-observation
    log-density evaluation: 2K+4 = 20 FP32 flop (SURVEY.md section 8d).
    FP32-pipe kernel: bound by the FP32 pipe, achieved = 20 flop/eval over the launch time.
    tcgen05 kernel: the contraction runs on the tensor pipe as 3xTF32 -- per 128-chain x group tile
    and sweep, 4 MMAs (A_hi.X_hi, A_lo.X_hi, A_hi.X_lo, 1.NE) of 2*128*Np*8 flop, Np = the group's
    observations rounded up to 16 -- and that pipe is the one that binds once latencies are hidden,
    so achieved = those TF32 flop over the launch time against the pipe's measured MMA rate;
    `useful_frac` is the algorithmic 20 flop/eval over the same peak (the 3xTF32 split, the ne MMA
    and the padding are the price of FP32 accuracy on that pipe)."""
    G, R, K = args.groups, args.obs, args.coef
    scale = chains / 1024.0
    if K == 0:
        # C5.  The kernel executes one ex2 per evaluation and one lg2 per fold of up to 64 observations (logarithm
        # of the product of the factors): with 50 trials per group 1 + 1/50 = 1.02 MUFU per evaluation ->
        # `achieved` / `frac` are that EXECUTED rate over the measured MUFU peak.  SURVEY.md section 8d's algorithmic figure (2 MUFU per evaluation: ex2 + lg2)
        # is reported beside it as `frac_at_survey_2_mufu_per_eval`.
        evals = 2.0 * G * R * chains
        perEval = 1.0 + float(-(-R // 64)) / R                      # one ex2 per observation, one lg2 per fold of 64
        executed = perEval * evals / (sweepMs * 1e-3)
        return {"bound": "mufu", "kernel": "sweep_kernel<Logit,2,float>", "achieved": executed / 1e9, "peak": peakMufu / 1e9,
                "unit": "Gop/s", "frac": executed / peakMufu, "mufu_executed_per_eval": perEval,
                "frac_at_survey_2_mufu_per_eval": 2.0 * evals / (sweepMs * 1e-3) / peakMufu,
                "traffic": TRAFFIC["c5"][0] * chains / 4096.0, "traffic_source": TRAFFIC["c5"][1],
                "fp32_pipe_peak_tflops": peakFp32 / 1e12,
                "peak_source": "MUFU pipe limit measured in this run by an ex2-only microbenchmark (mcmcn_peak_mufu); "
                               "nominal 148 SM x 16 lanes x 1.965 GHz = 4653"}
    P, N = K + 1, G * R
    algFlops = (2.0 * K + 4.0) * P * N * chains
    algTflops = algFlops / (sweepMs * 1e-3) / 1e12
    key = "tc" if tensorCore else "pipe"
    common = {"flop_per_eval": 2.0 * K + 4.0, "algorithmic_fp32_tflops": algTflops,
              "fp32_pipe_peak_tflops": peakFp32 / 1e12, "mufu_peak_gops": peakMufu / 1e9,
              "traffic": TRAFFIC[key][0] * scale,
              "traffic_source": TRAFFIC[key][1] + ", scaled by chains / 1,024; not measured live"}
    if not tensorCore:
        common.update({"bound": "fp32", "kernel": "sweep_kernel<LinReg<8>,4,float>", "achieved": algTflops,
                       "peak": peakFp32 / 1e12, "unit": "TFLOP/s", "frac": algFlops / (sweepMs * 1e-3) / peakFp32,
                       "peak_source": "FP32 pipe limit measured in this run by an FFMA-only microbenchmark "
                                      "(mcmcn_peak_fp32); MEASURED_PEAKS.json has no FP32 figure; nominal 74.4"})
        return common
    npad = max(16, (R + 15) // 16 * 16)
    tiles = ((chains + 127) // 128) * G * P
    kBlocks = 1 if K <= 8 else 2                                    # 3 MMAs per block of 8 coefficients + the ne MMA
    tf32Flops = tiles * (3 * kBlocks + 1) * 2.0 * 128 * npad * 8
    common.update({"bound": "tensor", "kernel": "sweep_tc_kernel (tcgen05.mma kind::tf32, 3xTF32 + ne)",
                   "achieved": tf32Flops / (sweepMs * 1e-3) / 1e12, "peak": peakTf32 / 1e12, "unit": "TFLOP/s",
                   "frac": tf32Flops / (sweepMs * 1e-3) / peakTf32,
                   "useful_frac": algFlops / (sweepMs * 1e-3) / peakTf32,
                   "tf32_flop_per_eval": tf32Flops / (P * N * chains),
                   "peak_source": "tensor pipe limit for this MMA shape (M128 N208 K8 kind::tf32, A in TMEM) measured "
                                  "in this run by an MMA-only microbenchmark (mcmcn_peak_tf32); MEASURED_PEAKS.json "
                                  "has bf16 only (1658 TFLOP/s burst; TF32 runs at half the bf16 rate = 829)"})
    return common


# ----------------------------------------------------------------------------- GPU arm
class Gpu(object):
    """Process-wide plumbing of the GPU arm: rank / world, device, barrier, max over ranks."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.group = dist.group.WORLD if self.world > 1 else None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def maxOverRanks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]


def peaks(eng, tensorCore):
    import ctypes
    import mcmcn_native as nat
    lib = nat.load()
    out = []
    for fn, wanted in (("mcmcn_peak_fp32", True), ("mcmcn_peak_mufu", True), ("mcmcn_peak_tf32", tensorCore)):
        v = ctypes.c_double(0.0)
        if wanted:
            nat.check(getattr(lib, fn)(ctypes.byref(v), eng.stream))
        out.append(v.value)
    return out


def dumpOutputs(directory, eng, store, row0):
    """What the timed path computed in its last step, as <directory>/<name>.npy: the rows it retained
    (`samples`, [row][column][chain], the store's float32) and the chain state it left, as Engine.getState
    names it (`theta`, `scale`, `lprior` [parameter][group][chain], `ll` [group][chain], `mu`, `sigma2`
    [parameter][chain] under partial pooling; float64).  The chains are a fixed, seeded sample (in chain
    order) where all of them would exceed DUMP_BYTES; the same arguments give the same sample."""
    import torch
    n = eng.nChains
    rows = store.tensor[row0:len(store.iterations)]
    state = [("theta", eng.theta), ("scale", eng.scale), ("lprior", eng.lprior), ("ll", eng.ll)]
    perChain = rows[..., 0].numel() * rows.element_size() + sum(t[..., 0].numel() * 8 for _, t in state)
    if eng.partial:
        perChain += 2 * eng.P * 8
    keep = min(n, max(1, DUMP_BYTES // perChain))
    chains = numpy.arange(n) if keep == n else numpy.sort(numpy.random.RandomState(0).choice(n, keep, replace=False))
    idx = torch.from_numpy(chains).to(eng.device)

    def pick(t):
        return t.index_select(t.dim() - 1, idx).cpu().numpy()
    out = dict((name, pick(t)) for name, t in state)
    out["samples"] = pick(rows)
    if eng.partial:
        hyper = pick(eng.hyper)
        out["mu"], out["sigma2"] = hyper[0], hyper[1]
    os.makedirs(directory, exist_ok=True)
    for name, arr in out.items():
        numpy.save(os.path.join(directory, name + ".npy"), arr)


def stepPass(gpu, args, chains, chainId0, withClocks, diagnostics=False, dumpDir=None):
    """W warm-up + K timed steps of args.iters_per_step iterations with everything resident in HBM.
    Returns a dict: ms (max over ranks), per-kernel timing, roofline inputs, optionally the timed
    between-chain diagnostics of the retained rows.  With `dumpDir`, rank 0 writes what the last
    timed step computed there (dumpOutputs)."""
    torch = gpu.torch
    from engine import Engine, SampleStore, retainedCount
    from objectives import Objective
    G, R, K = args.groups, args.obs, args.coef
    if K == 0:
        x, y, names, ranges = makeLogitWorkload(G, R)
        obj = Objective.bernoulli_logit(x, y, args.precision)
    else:
        X, y, names, ranges = makeWorkload(G, R, K)
        obj = Objective.linear_regression(X, y, args.precision)
    eng = Engine(obj, G, R, args.pooling, chains, priorDistribution=fixedPriors(args.pooling, K),
                 chainId0=chainId0, seed=args.seed)
    eng.initialise(names, ranges)
    ips = args.iters_per_step
    total = (args.warmup + args.steps) * ips
    burn, thin = total // 2, args.thin
    nRows = len([i for i in range(total) if i % thin == 0 and i >= burn])
    store = SampleStore(eng, max(nRows, 1), torch.float32)
    tensorCore = eng.usesTensorCore
    peakFp32, peakMufu, peakTf32 = peaks(eng, tensorCore)

    for w in range(args.warmup):
        eng.run(w * ips, ips, burn, thin, store=store)
    gpu.barrier()
    sampler = ClockSampler(gpu.local) if (withClocks and gpu.rank == 0) else None
    timing = numpy.zeros(12)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for k in range(args.steps):
        eng.run((args.warmup + k) * ips, ips, burn, thin, store=store, timing=timing)
    ev1.record()
    gpu.barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if sampler else None
    eng.collectTiming()            # durations of the launches sampled (every 8th iteration) inside the timed region
    ms = gpu.maxOverRanks([ms])[0]
    if dumpDir is not None and gpu.rank == 0:
        last = (args.warmup + args.steps - 1) * ips
        dumpOutputs(dumpDir, eng, store, len(store.iterations) - retainedCount(last, last + ips, burn, thin))
    sweepMs = timing[0] / max(timing[6], 1.0)
    out = {"ms": ms, "chains": chains, "P": len(names), "N": G * R, "clocks": clocks,
           "launches": int(timing[3] + timing[4] + timing[5]),
           "kernel_ms": {"step_kernel_avg": sweepMs, "hyper_kernel_avg": timing[1] / max(timing[7], 1.0),
                         "writeback_avg": timing[2] / max(timing[8], 1.0),
                         "timed_launches": int(timing[6] + timing[7] + timing[8]),
                         "step_kernel_share": sweepMs * timing[3] / ms},
           "roofline": roofline(args, tensorCore, sweepMs, chains, peakFp32, peakTf32, peakMufu),
           "rows": len(store.iterations)}
    if diagnostics and len(store.iterations) >= 6:
        out["diagnostics"] = storeDiagnostics(gpu, store, chains)
    del store, eng
    torch.cuda.empty_cache()
    return out


def storeDiagnostics(gpu, store, chains):
    """Between-chain diagnostics of the rows a step pass retained, on the device.  With N > 1 the half-chain
    moments and per-lag sums cross NVLink in one NCCL all-gather per slab of columns (R-hat / ESS), and the
    pooled median / HDI take a key-partitioned all-to-all: the path's only collectives, timed here."""
    torch = gpu.torch
    from sampleDiagnosis import convergenceFromStore, orderStatisticsFromStore
    nKept = len(store.iterations)
    if gpu.world > 1:
        # warm the communicator up for both patterns (NCCL sets its peer-to-peer channels up at the first
        # all-to-all: seconds, once per process), on a few columns and outside the timed region
        few = store.tensor[:, :min(8 * gpu.world, store.tensor.shape[1])].contiguous()
        convergenceFromStore(few, nKept, chains, group=gpu.group)
        orderStatisticsFromStore(few, nKept, chains, group=gpu.group)
        del few
    gpu.barrier()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    info = {}
    e[0].record()
    rhat, ess = convergenceFromStore(store.tensor, nKept, chains, group=gpu.group, timing=info)
    e[1].record()
    stats = orderStatisticsFromStore(store.tensor, nKept, chains, group=gpu.group, timing=info)
    e[2].record()
    gpu.barrier()
    msConv, msOrder = gpu.maxOverRanks([e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])])
    fin = torch.isfinite(ess)
    return {"rows": nKept, "half_chains": 2 * chains * gpu.world, "keys": int(ess.numel()),
            "min_ess": float(ess[fin].min()) if bool(fin.any()) else None,
            "max_rhat": float(rhat[torch.isfinite(rhat)].max()),
            "median_of_first_key": float(stats[0, 0]),
            "rhat_ess_ms": msConv, "median_hdi_ms": msOrder, "diag_ms": msConv + msOrder,
            "all_gather_bytes_per_rank": int(info.get("gathered_bytes", 0)),
            "all_to_all_bytes_per_rank": int(info.get("exchanged_bytes", 0)),
            "note": "rows retained by the timed steps only (a slice of the schedule: not converged, see full_run "
                    "for the whole config); times are max over ranks, CUDA events"}


def fullRun(gpu, args, chainsTotal, nIter, nSamples, withDiagnostics):
    """The configuration through the reference's own calls, host arrays in, files out:
    samplePosterior(...) -> sample/samples[.rank<r>].npy + manifest.json, then sampleDiagnosis.Diagnostic
    over those files (R-hat, ESS of every column).  Wall-clock, barrier on both sides, max over ranks."""
    torch = gpu.torch
    import posteriorSampling as ps
    import sampleDiagnosis as sd
    from objectives import Objective
    G, R, K = args.groups, args.obs, args.coef
    X, y, names, ranges = makeWorkload(G, R, K)                       # host numpy arrays: what a user holds
    # where the store goes: the first of /dev/shm and the temp directory with room for it (never the source tree,
    # which may be read-only); if neither has, fewer retained rows (said in the record) rather than a failed run
    elem = 8 if args.store_dtype == "float64" else 4
    rowBytes = (K + 1) * (G + 2) * chainsTotal * elem
    need = nSamples * rowBytes
    roots = [args.output_root] if args.output_root else ["/dev/shm", tempfile.gettempdir()]
    free = []
    for cand in roots:
        try:
            os.makedirs(cand, exist_ok=True)
            free.append((shutil.disk_usage(cand).free, cand))
        except OSError:
            continue
    fits = [c for f, c in free if f >= 1.05 * need + (1 << 30)]
    reduced = None
    if fits:
        base = fits[0]
    else:
        room, base = max(free) if free else (0, tempfile.gettempdir())
        reduced = max(4, int(0.8 * room // max(rowBytes, 1)) // 2 * 2)
        nSamples = min(nSamples, reduced)
    if gpu.world > 1:                                   # one decision for all ranks (rank 0's)
        choice = [base, nSamples, reduced]
        gpu.dist.broadcast_object_list(choice, src=0)
        base, nSamples, reduced = choice
    out = os.path.join(base, "mcmcn_bench_%s" % (os.environ.get("MASTER_PORT", "0") if gpu.world > 1 else os.getpid()))
    ps.CSV_VALUE_LIMIT = 0                                             # binary store
    ps.STORE_DTYPE = args.store_dtype
    gpu.barrier()
    t0 = time.perf_counter()
    handle = Objective.linear_regression(X, y, args.precision)
    ps.samplePosterior(chainsTotal, nIter, nSamples, names, G, R, args.pooling, handle, out,
                       saveLogLikelihood=False, startingPointValueRange=ranges, displayProgress=False)
    gpu.barrier()
    wall = gpu.maxOverRanks([time.perf_counter() - t0])[0]
    run = ps.lastRun
    eng, store = run["engine"], run["store"]
    rows = len(run["retained"])
    myChains = run["chains"][1] - run["chains"][0]
    d2h = rows * eng.nCol * eng.S * elem
    h2d = int(eng.stepInput.numel() * eng.stepInput.element_size() + eng._data.numel() * eng._data.element_size()
              + 3 * 8 * eng.P * eng.G * eng.S)                         # observation blocks + the start state
    rec = {"call": "posteriorSampling.samplePosterior(nChains=%d, nIter=%d, nSamples=%d, ..., saveLogLikelihood=False)"
                   % (chainsTotal, nIter, nSamples),
           "chains": chainsTotal, "iterations": nIter, "retained_rows": rows, "wall_s": wall,
           "sampling_loop_s": gpu.maxOverRanks([run["sampling_seconds"]])[0],
           "chain_iterations_per_s": chainsTotal * nIter / wall,
           "store": {"dtype": args.store_dtype, "bytes_per_rank": int(rows * eng.nCol * myChains * elem),
                     "directory": base, "device_ring_bytes": int(run["store_device_bytes"]),
                     "pinned_host_bytes": int(run.get("store_pinned_bytes", run["store_device_bytes"]))},
           "phases_s": {k: round(v, 3) for k, v in run.get("phases", {}).items()},
           "h2d_bytes": h2d, "d2h_bytes": int(d2h)}
    if reduced is not None:
        rec["store"]["note"] = "nSamples cut to %d: no directory with room for the configured store" % nSamples
    del eng, store
    ps.lastRun = None
    torch.cuda.empty_cache()
    if withDiagnostics:
        gpu.barrier()
        t1 = time.perf_counter()
        diag = sd.Diagnostic(out + "/sample/")                          # sharded: one shard per rank + NCCL exchanges
        rhat = numpy.array([diag.rhat[k] for k in diag._keys])
        ess = numpy.array([diag.effectiveN[k] for k in diag._keys])
        gpu.barrier()
        diagS = gpu.maxOverRanks([time.perf_counter() - t1])[0]
        fin = numpy.isfinite(ess)
        rec["diagnostics"] = {"call": "sampleDiagnosis.Diagnostic(outputDirectory + '/sample/') -> rhat, effectiveN, median, hdi",
                              "keys": int(ess.size), "half_chains": int(diag._m), "draws_per_half_chain": int(diag._n),
                              "max_rhat": float(numpy.nanmax(rhat)), "max_rhat_key": diag._keys[int(numpy.nanargmax(rhat))],
                              "share_rhat_below_1.1": float(numpy.mean(rhat < 1.1)),
                              "keys_rhat_above_1.1": [diag._keys[i] for i in numpy.nonzero(~(rhat < 1.1))[0][:8]],
                              "min_ess_key": diag._keys[int(numpy.argmin(numpy.where(fin, ess, numpy.inf)))],
                              "min_ess": float(ess[fin].min()), "median_ess": float(numpy.median(ess[fin])),
                              "seconds": diagS}
        rec["min_ess_per_s"] = rec["diagnostics"]["min_ess"] / wall
        rec["min_ess_per_s_note"] = "min over all keys of Diagnostic.effectiveN (sampleDiagnosis.py:232-255) / wall time " \
                                    "of the samplePosterior call (start-up, burn-in, sampling, writing the store)"
    gpu.barrier()
    if gpu.rank == 0:
        shutil.rmtree(out, ignore_errors=True)
    return rec


def runGpu(args):
    gpu = Gpu()
    torch = gpu.torch
    world, rank = gpu.world, gpu.rank
    if world > 1 and args.workload == "c3":                # config 4: 16,384 chains in total, sharded
        chains = C4_CHAINS // world
    else:
        chains = args.chains_per_gpu
    main = stepPass(gpu, args, chains, rank * chains, withClocks=True, diagnostics=True, dumpDir=args.dump_outputs)
    P, N = main["P"], main["N"]
    chainIters = world * chains * args.iters_per_step * args.steps
    value = chainIters / (main["ms"] * 1e-3)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms"] / args.steps,
            "higher_is_better": True, "scaling": "weak" if world == 1 else "strong", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "f64", "data": "synthetic",
            "config": workloadConfig(args, chains, world),
            "evals_per_sec": value * P * N, "evals_per_sec_per_gpu": value * P * N / world,
            "gpu_launches": main["launches"], "kernel_ms": main["kernel_ms"], "roofline": main["roofline"],
            "clocks": main["clocks"], "diagnostics": main.get("diagnostics")}

    # ---- e2e: the configuration through samplePosterior, host arrays in, sample files out
    full = None
    if args.coef and not args.no_full_run:
        try:
            if world == 1:
                full = fullRun(gpu, args, chains, args.full_iters, args.full_samples, withDiagnostics=True)
            else:
                full = fullRun(gpu, args, C4_CHAINS, args.c4_iters, args.c4_samples, withDiagnostics=True)
        except Exception as err:                        # the line is still printed, with the failure in it
            import traceback
            traceback.print_exc()
            line["full_run"] = {"error": "%s: %s" % (type(err).__name__, err)}
    if full is not None:
        stepsEq = full["iterations"] / float(args.iters_per_step)
        line["e2e"] = {"value": full["chain_iterations_per_s"], "unit": UNIT,
                       "h2d_bytes_per_step": int(full["h2d_bytes"] / stepsEq), "d2h_bytes_per_step": int(full["d2h_bytes"] / stepsEq),
                       "what": "one samplePosterior call on host arrays (%d chains x %d iterations, %d retained rows per chain "
                               "streamed through pinned memory into sample/*.npy): chains x iterations / wall time of the call; "
                               "bytes per step = the call's bytes per %d iterations" % (full["chains"], full["iterations"],
                                                                                        full["retained_rows"], args.iters_per_step)}
        line["full_run"] = full
    else:
        line["e2e"] = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                       "what": "skipped (--no-full-run)" if args.no_full_run or not args.coef else "failed, see full_run.error"}

    # ---- sub-records (one GPU): config 4's single-GPU point and config 5
    if world == 1 and args.workload == "c3" and not args.no_sub_records:
      try:
        sub = argparse.Namespace(**vars(args))
        sub.steps, sub.warmup = 5, 3
        c4 = stepPass(gpu, sub, C4_CHAINS, 0, withClocks=False, diagnostics=True)
        line["c4_single_gpu"] = {"chains": C4_CHAINS, "value": C4_CHAINS * sub.iters_per_step * sub.steps / (c4["ms"] * 1e-3),
                                 "unit": UNIT, "steps": sub.steps, "warmup": sub.warmup, "kernel_ms": c4["kernel_ms"],
                                 "roofline_frac": c4["roofline"]["frac"], "diagnostics": c4.get("diagnostics")}
        for pooling in ("partial", "none"):
            c5 = argparse.Namespace(**vars(args))
            c5.groups, c5.obs, c5.coef, c5.pooling = 10000, 50, 0, pooling
            c5.iters_per_step, c5.thin, c5.steps, c5.warmup = 20, 20, 5, 3
            r5 = stepPass(gpu, c5, 4096, 0, withClocks=False)
            v5 = 4096 * c5.iters_per_step * c5.steps / (r5["ms"] * 1e-3)
            line["c5_" + pooling] = {"workload": workloadConfig(c5, 4096)["workload"], "chains": 4096, "value": v5, "unit": UNIT,
                                     "evals_per_sec": v5 * 2 * 500000, "steps": c5.steps, "warmup": c5.warmup,
                                     "iters_per_step": c5.iters_per_step, "kernel_ms": r5["kernel_ms"], "roofline": r5["roofline"]}
      except Exception as err:
        import traceback
        traceback.print_exc()
        line["sub_records_error"] = "%s: %s" % (type(err).__name__, err)

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpuBaselineRecord(args)
            except Exception as err:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "reference", "sample": "failed: %s" % err}
        emit(json.dumps(line))
    if world > 1:
        gpu.dist.destroy_process_group()


_REAL_STDOUT = None


def emit(text):
    """The one JSON line, on the process's real stdout."""
    if _REAL_STDOUT is None:
        print(text, flush=True)
    else:
        os.write(_REAL_STDOUT, (text + "\n").encode())


def main():
    global _REAL_STDOUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c3", "c5"],
                    help="c3 (default, the config BASELINE.json's metric is quoted on; with --gpus N > 1 config 4: 16,384 "
                         "chains in total) or c5 (Bernoulli-logit: 10,000 groups x 50 trials, 4,096 chains)")
    ap.add_argument("--chains-per-gpu", type=int, default=1024)
    ap.add_argument("--groups", type=int, default=1024)
    ap.add_argument("--obs", type=int, default=200)
    ap.add_argument("--coef", type=int, default=8)
    ap.add_argument("--iters-per-step", type=int, default=50)
    ap.add_argument("--thin", type=int, default=10)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp64"])
    ap.add_argument("--pooling", default="partial", choices=["partial", "none"],
                    help="partial (default, the BASELINE metric's mode) or none (BASELINE config 5 names both)")
    # the whole configuration through samplePosterior (e2e / full_run)
    ap.add_argument("--full-iters", type=int, default=20000, help="config 3: 20k iterations")
    ap.add_argument("--full-samples", type=int, default=1000, help="retained rows per chain (burn 10,000, thin 10)")
    ap.add_argument("--c4-iters", type=int, default=20000, help="N > 1: iterations of the samplePosterior call on config 4 (config 3's 20k)")
    ap.add_argument("--c4-samples", type=int, default=100, help="retained rows per chain (burn 10,000, thin 100: a 60 GB FP32 store; "
                                                                "config 3's 1,000 rows x 16,384 chains would be 605 GB)")
    ap.add_argument("--store-dtype", default="float32", choices=["float32", "float64"],
                    help="sample store of the full run (float32 is the store's documented opt-in: 37.8 GB for config 3)")
    ap.add_argument("--output-root", default=None, help="where the full run writes (default /dev/shm, else the temp dir)")
    ap.add_argument("--no-full-run", action="store_true")
    ap.add_argument("--no-sub-records", action="store_true")
    # CPU arms
    ap.add_argument("--cpu-iters", type=int, default=40, help="oracle port: iterations of the cpu_baseline sample")
    ap.add_argument("--port-iters", type=int, default=5, help="--impl reference without baseline/_ref: port iterations per step")
    ap.add_argument("--ref-iters", type=int, default=6, help="unmodified reference: iterations per step (>= 6)")
    ap.add_argument("--ref-groups", type=int, default=64, help="unmodified reference: groups of the per-step sample")
    ap.add_argument("--port", action="store_true", help="--impl reference: time the oracle port even if baseline/_ref is staged")
    ap.add_argument("--ref-calibration-iters", type=int, default=30,
                    help="--impl reference: iterations of the two runs on ALL groups (one process; one process per core)")
    ap.add_argument("--no-calibration", action="store_true", help="--impl reference: skip the two full-shape runs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (retained rows and chain state of a "
                         "seeded sample of rank 0's chains) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs is not None and (args.impl != "b200" or args.steps < 1):
        ap.error("--dump-outputs needs the GPU arm (--impl b200) and --steps >= 1")
    # Everything libraries print on file descriptor 1 (NCCL's version banner under NCCL_DEBUG=VERSION,
    # for one) goes to stderr; stdout carries the JSON line and nothing else.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.workload == "c5":
        args.groups, args.obs, args.coef, args.chains_per_gpu = 10000, 50, 0, 4096
        args.iters_per_step, args.thin = min(args.iters_per_step, 20), max(args.thin, 20)
        args.ref_groups = min(args.ref_groups * 10, args.groups)
    args.ref_groups = min(args.ref_groups, args.groups)
    if args.warmup < 3 and args.impl == "b200":
        print("warning: the timing rules ask for >= 3 warm-up steps", file=sys.stderr)
    if args.impl == "reference":
        runReference(args)
    else:
        runGpu(args)


if __name__ == "__main__":
    main()
