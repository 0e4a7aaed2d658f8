"""Drop-in for the reference's ``posteriorSampling`` module: same ``samplePosterior``
signature and outputs (/root/reference/posteriorSampling.py:28-216), but every chain is
advanced together on the GPU by the CUDA step kernels behind the C ABI (include/mcmcn.h).

What changes on purpose (BASELINE.json north star):
  * ``logLikelihoodFunction`` must be an ``objectives.Objective`` handle (a device function
    from the registry, or NVRTC-compiled source).  A Python callable raises TypeError; there is
    no CPU fallback.
  * ``nProcesses`` is accepted and ignored: chains are GPU threads, not OS processes.
  * proposals / accept uniforms come from per-chain Philox streams keyed by the global chain id
    (the reference uses numpy's global MT19937, seed = chain); start states still come from each
    chain's MT19937 stream in the reference's order, so they equal the reference's.
  * at scale the retained samples stream into a binary store (``sample/samples[.rank<r>].npy`` +
    ``sample/manifest.json``, one shard file per rank) that ``sampleDiagnosis`` reads; at example scale
    the reference's ``sample.<chain>.csv`` / ``logLikelihood.<chain>.csv`` files are written.
Under ``torch.distributed`` (one process per GPU) the chains are split contiguously over the
ranks; sampling needs no communication.
"""

import datetime
import time
import json
import logging
import os
import shutil

import numpy
import torch

from engine import Engine, SampleStore, burnThin, retainedIterations
from mcmcn_native import _rankWorld, chainRange
from objectives import Objective

# above this many retained values (rows x columns x chains) the samples go to the binary store
CSV_VALUE_LIMIT = int(os.environ.get("MCMCN_CSV_LIMIT", 20000000))
# the pointwise log-likelihood output is refused above this many values (rows x N x chains)
LOGLIK_VALUE_LIMIT = int(os.environ.get("MCMCN_LOGLIK_LIMIT", 200000000))
# the binary store keeps the chains' FP64 values; "float32" (6e-8 relative, below the reference's "%f"
# for |values| < 16) is an explicit opt-in that the manifest records
STORE_DTYPE = os.environ.get("MCMCN_STORE_DTYPE", "float64")


def samplePosterior(nChains, nIter, nSamples,
                    parameterName, nGroups, nResponsesPerGroup,
                    pooling, logLikelihoodFunction,
                    outputDirectory,
                    saveLogLikelihood=True,
                    priorDistribution=None,
                    startWithMLE=False, startingPointValueRange=None,
                    nProcesses=1, displayProgress=True, loggingLevel="info"):
    """Samples from the posterior distribution; samples are saved under ``outputDirectory``
    (see the reference's docstring, posteriorSampling.py:36-144, for the arguments)."""
    startTime = datetime.datetime.now()
    rank, world = _rankWorld()

    # argument errors are raised identically on every rank, before the first collective
    if not isinstance(logLikelihoodFunction, Objective):
        raise TypeError("logLikelihoodFunction must be an objectives.Objective handle (a device function); "
                        "Python callables cannot run on the GPU and there is no CPU fallback")
    if pooling not in ("partial", "none", "complete"):             # :1040-1043
        raise Exception("Invalid pooling: ", pooling)
    burn, thin = burnThin(nIter, nSamples)                          # :1018-1027
    if nChains < world:
        raise ValueError("fewer chains (%d) than ranks (%d)" % (nChains, world))

    if rank == 0:
        if os.path.exists(outputDirectory):
            shutil.rmtree(outputDirectory)                         # :149-150
    _barrier(world)
    sampleDirectory = outputDirectory + "/sample/"
    os.makedirs(sampleDirectory, exist_ok=True)
    logDirectory = outputDirectory + "/log/"
    os.makedirs(logDirectory, exist_ok=True)

    logger = _getLogger(logDirectory + "samplePosterior.log", "samplePosterior", loggingLevel)
    msg = "MCMC sampling.\n"
    msg += "\tpooling: %s.\n" % pooling
    msg += "\tnChains: %i, nIterPerChain: %i, nSamplesPerChain: %i." % (nChains, nIter, nSamples)
    logger.info(msg)
    if displayProgress and rank == 0:
        print(msg)

    # a rank that fails between here and the closing barrier tells its peers, so that nobody waits forever
    failure = None
    try:
        elapsed = _sampleShard(rank, world, nChains, nIter, burn, thin, parameterName, nGroups, nResponsesPerGroup,
                               pooling, logLikelihoodFunction, sampleDirectory, logDirectory, saveLogLikelihood,
                               priorDistribution, startWithMLE, startingPointValueRange, displayProgress,
                               loggingLevel, logger)
    except BaseException as err:        # noqa: B902 -- re-raised below, after the peers know
        failure = err
    if world > 1:
        import torch.distributed as dist
        flag = torch.tensor([0 if failure is None else 1], dtype=torch.int32,
                            device="cuda" if dist.get_backend() == "nccl" else "cpu")
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if failure is None and int(flag[0]):
            failure = RuntimeError("samplePosterior failed on another rank")
    if failure is not None:
        raise failure

    endTime = datetime.datetime.now()
    msg = "Finished. The elapsed time in total is %s." \
        % datetime.timedelta(seconds=int((endTime - startTime).total_seconds()))
    logger.info(msg)
    if displayProgress and rank == 0:
        print("")
        _printProgress(msg)


def _sampleShard(rank, world, nChains, nIter, burn, thin, parameterName, nGroups, nResponsesPerGroup, pooling,
                 objective, sampleDirectory, logDirectory, saveLogLikelihood, priorDistribution, startWithMLE,
                 startingPointValueRange, displayProgress, loggingLevel, logger):
    """This rank's chains (contiguous global ids; Philox and the start-state streams are keyed by them):
    start state, Sampler._loop (:862-896), sample files."""
    lo, hi = chainRange(nChains, rank, world)
    myChains = hi - lo
    show = displayProgress and rank == 0
    phases, mark = {}, [time.perf_counter()]

    def phase(name):                                               # wall seconds of the call's phases, kept in lastRun
        now = time.perf_counter()
        phases[name] = phases.get(name, 0.0) + now - mark[0]
        mark[0] = now

    eng = Engine(objective, nGroups, nResponsesPerGroup, pooling, myChains,
                 priorDistribution=priorDistribution, chainId0=lo,
                 seed=int(os.environ.get("MCMCN_SEED", "0")))
    chainLoggers = [_getLogger(logDirectory + "/mcmc.chain%.2i.log" % c, "mcmc.chain%.2i" % c, loggingLevel)
                    for c in range(lo, hi)] if myChains <= 64 else []
    if pooling == "partial" and priorDistribution is not None:
        logger.info("Partial pooling ignores prior distribution.")  # :713-714
    phase("engine")
    _progress(logger, show, "Started looking for a reasonable starting state.")
    eng.initialise(parameterName, startingPointValueRange, startWithMLE, logger)
    _progress(logger, show, "Found a reasonable starting state.")
    phase("start_state")

    retained = retainedIterations(nIter, burn, thin)
    nValues = len(retained) * eng.nCol * nChains
    useCsv = nValues <= CSV_VALUE_LIMIT
    if saveLogLikelihood and len(retained) * eng.nObservations * nChains > LOGLIK_VALUE_LIMIT:
        raise ValueError("saveLogLikelihood=True would write %d x %d x %d log-likelihood values; pass "
                         "saveLogLikelihood=False (or raise MCMCN_LOGLIK_LIMIT)"
                         % (len(retained), eng.nObservations, nChains))

    def appendLogLikelihood(row0, block):                          # block [rows][N][myChains], in row order
        for c in range(myChains):                                   # Sampler._printLogLikelihood, :907-909
            with open(sampleDirectory + "/logLikelihood.%i.csv" % (lo + c), "a") as h:
                for r in range(block.shape[0]):
                    h.write(",".join(["%f" % v for v in block[r, :, c]]))
                    h.write("\n")

    # Example scale: every row stays on the device and the reference's CSV files are written at the end.
    # At scale: the rows stream through a two-chunk ring on the device into a .npy file per rank.
    storeDtype = torch.float64
    if not useCsv and STORE_DTYPE == "float32":
        storeDtype = torch.float32
    shardFile = "samples.npy" if world == 1 else "samples.rank%d.npy" % rank
    store = SampleStore(eng, max(len(retained), 1), storeDtype,
                        path=None if useCsv else os.path.join(sampleDirectory, shardFile),
                        logLikelihood=bool(saveLogLikelihood), logLikSink=appendLogLikelihood)

    # ---- Sampler._loop (:862-896): one call per progress mark; the store splits it where a chunk is full
    stops = set([nIter])
    loggingInterval = int(numpy.round(nIter / 10.))
    if loggingInterval > 0:
        stops.update(range(loggingInterval, nIter, loggingInterval))
    phase("store")
    loopStart = datetime.datetime.now()
    _progress(logger, show, r"Sampling started. 0% complete.")
    cur = 0
    for stop in sorted(stops):
        eng.run(cur, stop - cur, burn, thin, store=store)
        cur = stop
        if loggingInterval > 0 and stop % loggingInterval == 0 and stop < nIter:
            torch.cuda.synchronize()
            now = datetime.datetime.now()
            percentage = float(stop) / nIter
            remain = (1 - percentage) * (now - loopStart) / percentage
            _progress(logger, show, "%i%% complete. ETA: %s." % (percentage * 100, _getStrfTime(now + remain)))
    torch.cuda.synchronize()
    elapsed = datetime.datetime.now() - loopStart
    _progress(logger, show, "100%% complete. Elapsed Time: %s."
              % datetime.timedelta(seconds=int(elapsed.total_seconds())))

    phase("sampling_loop")
    phases["waited_for_store_writers"] = store.waitedForWriters     # part of the sampling loop
    phases["retire_waited_for_device"] = store.retireWaitedForDevice
    phases["retire_wrote"] = store.retireWrote
    # ---- outputs
    store.finish()
    phase("store_drain")
    header = sampleHeader(parameterName, eng.G, pooling)
    if useCsv:
        rows = store.hostArray()                                    # [rows][ncol][myChains]
        for c in range(myChains):
            writeSampleCsv(sampleDirectory + "/sample.%i.csv" % (lo + c), lo + c, header,
                           retained, rows[:, :, c])
    for c, lg in enumerate(chainLoggers):
        lg.info("chain %i. 100%% complete. Elapsed Time: %s."
                % (lo + c, datetime.timedelta(seconds=int(elapsed.total_seconds()))))
    global lastRun
    lastRun = {"engine": eng, "store": store, "retained": retained, "chains": (lo, hi),
               "sampling_seconds": elapsed.total_seconds(), "store_device_bytes": store.deviceBytes,
               "store_pinned_bytes": store.deviceBytes if store.streamed else 0,    # two chunks, as on the device
               "phases": phases}
    _barrier(world)                                                 # every shard file is complete
    if not useCsv and rank == 0:
        writeManifest(sampleDirectory, header, retained, nChains, world, pooling,
                      "float64" if storeDtype == torch.float64 else "float32")
    phase("files")
    return elapsed


# What the last samplePosterior call of this process left on the device (engine, store, timings): lets a
# caller that holds the process (bench.py, notebooks) run convergenceFromStore without re-reading files.
lastRun = None


# ------------------------------------------------------------------------------ output format
def sampleHeader(parameterName, nSteppedGroups, pooling):
    """Column names of a sample file (posteriorSampling.py:640-646, :771-778, :504-507, :263)."""
    cols = []
    for name in parameterName:
        if pooling == "partial":
            cols += ["%s_mu" % name, "%s_sigma2" % name]
        cols += ["%s[%.3i]" % (name, j) for j in range(nSteppedGroups)]
    return cols


def writeSampleCsv(path, chain, header, iterations, rows):
    """``sample.<chain>.csv`` exactly as Sampler._printHeader/_printSample write it (:898-905)."""
    with open(path, "w") as h:
        h.write("index,chain," + ",".join(header))
        h.write("\n")
        for i, row in zip(iterations, rows):
            h.write("%i,%i," % (i, chain))
            h.write(",".join(["%f" % v for v in row]))
            h.write("\n")


def writeManifest(sampleDirectory, header, iterations, nChains, world, pooling, dtype):
    """``sample/manifest.json``: what sampleDiagnosis.openSamples reads.  One shard file per rank, each
    [rows][columns][chains of that rank] (.npy), chains split contiguously over the ranks (chainRange)."""
    shards = [{"file": "samples.npy" if world == 1 else "samples.rank%d.npy" % r,
               "chains": list(chainRange(nChains, r, world))} for r in range(world)]
    man = {"format": "mcmcn-samples-2", "header": list(header), "iterations": list(map(int, iterations)),
           "nChains": int(nChains), "pooling": pooling, "dtype": dtype,
           "layout": "[rows][columns][chains]", "shards": shards}
    if dtype == "float32":
        man["note"] = "draws rounded to float32 on request (MCMCN_STORE_DTYPE=float32): 6e-8 relative"
    with open(os.path.join(sampleDirectory, "manifest.json"), "w") as h:
        json.dump(man, h)


# ------------------------------------------------------------------------------ plumbing
def _barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def _progress(logger, display, msg):
    logger.info(msg)
    if display:
        _printProgress(msg)


def _getLogger(logFile, logName, loggingLevel):
    """:1161-1182 (one handler per log file; the reference adds a handler on every call)."""
    level = {"debug": logging.DEBUG, "info": logging.INFO, "warning": logging.WARNING,
             "error": logging.ERROR}[loggingLevel]
    logger = logging.getLogger(logName)
    logger.setLevel(level)
    for hd in list(logger.handlers):
        logger.removeHandler(hd)
        hd.close()
    handler = logging.FileHandler(logFile)
    handler.setLevel(level)
    handler.setFormatter(logging.Formatter("%(asctime)s - %(name)s - %(levelname)s\n%(message)s\n"))
    logger.addHandler(handler)
    return logger


def _printProgress(msg):
    print(_getStrfTime(datetime.datetime.now()) + "\t" + msg)


def _getStrfTime(time):
    return time.strftime("%Y/%m/%d %H:%M:%S")
