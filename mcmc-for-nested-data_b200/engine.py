"""Host side of the GPU engine: model packing, chain state, start-up, run loop, sample store.

PyTorch is used for device memory, streams and (in the callers) torch.distributed only;
every kernel launch goes through the C ABI in include/mcmcn.h via mcmcn_native (ctypes).

Reference symbols this module stands in for (``/root/reference/posteriorSampling.py``):
  MCMC.__init__ / _findStartingPoint ....... :944-1095   -> Engine.initialise
  StepMethod.__init__ / _setStartingPoint .. :517-592, :725-758 -> Engine.initialise
  Sampler.sample / _loop .................... :827-896    -> Engine.run
"""

import ctypes
import os
import threading
import time

import numpy
import scipy.special
import torch

import mcmcn_native as nat
from mcmcn_native import _hostThreads, _ptr
from objectives import Objective

_NORM_PDF_LOGC = numpy.log(numpy.sqrt(2 * numpy.pi))


def burnThin(nIter, nSamples):
    """posteriorSampling.py:1018-1027."""
    if nIter < nSamples:
        print("nIter (%i) cannot be less than nSamples (%i)." % (nIter, nSamples))
        raise Exception()
    elif nIter // 2 > nSamples:
        burn = nIter // 2
    else:
        burn = nIter - nSamples
    thin = int(numpy.ceil((nIter - burn) / nSamples))
    return burn, thin


def _retainedRange(lo, hi, burn, thin):
    """Iterations i in [lo, hi) whose state Sampler._loop writes out: i >= burn and i % thin == 0 (:887)."""
    return range(-(-max(lo, burn) // thin) * thin, hi, thin)


def retainedIterations(nIter, burn, thin):
    """Iterations whose state Sampler._loop writes out (:887)."""
    return list(_retainedRange(0, nIter, burn, thin))


def hostNormLogpdf(x, loc, scale):
    """scipy.stats.norm(loc, scale).logpdf(x), same operation order (used for the start state)."""
    with numpy.errstate(all="ignore"):
        y = (x - loc) / scale
        out = -y ** 2 / 2.0 - _NORM_PDF_LOGC - numpy.log(scale)
        bad = ~(numpy.asarray(scale) > 0) | numpy.isnan(y)
        return numpy.where(bad, numpy.nan, out)


def priorFromScipy(frozen):
    """Map a frozen scipy.stats distribution (what the reference takes in
    ``priorDistribution``) to the device prior record."""
    name = frozen.dist.name
    shapes, loc, scale = frozen.dist._parse_args(*frozen.args, **frozen.kwds)
    pr = nat.Prior()
    pr.loc, pr.scale = float(loc), float(scale)
    with numpy.errstate(all="ignore"):
        pr.log_scale = float(numpy.log(float(scale)))
    pr.a, pr.c0, pr.b = 0.0, 0.0, 0.0
    # every constant below is formed exactly as scipy's _logpdf forms it, so that the device value
    # differs from frozen.logpdf only by the rounding of log / log1p / exp
    if name == "norm":
        pr.family = nat.PRIOR_NORM
    elif name == "gamma":
        pr.family = nat.PRIOR_GAMMA
        pr.a = float(shapes[0])
        pr.c0 = float(scipy.special.gammaln(pr.a))
    elif name == "uniform":
        pr.family = nat.PRIOR_UNIFORM
    elif name == "expon":
        pr.family = nat.PRIOR_EXPON
    elif name == "halfnorm":
        pr.family = nat.PRIOR_HALFNORM
    elif name == "lognorm":
        pr.family = nat.PRIOR_LOGNORM
        pr.a = float(shapes[0])
        pr.c0 = float(2 * pr.a ** 2)
    elif name == "cauchy":
        pr.family = nat.PRIOR_CAUCHY
    elif name == "t":
        pr.family = nat.PRIOR_T
        pr.a = float(shapes[0])
        if not numpy.isfinite(pr.a):
            raise ValueError("t prior with df = inf: use norm")
        pr.c0 = float(numpy.log(scipy.special.poch(0.5 * pr.a, 0.5)) - 0.5 * (numpy.log(pr.a) + numpy.log(numpy.pi)))
    elif name == "beta":
        pr.family = nat.PRIOR_BETA
        pr.a, pr.b = float(shapes[0]), float(shapes[1])
        pr.c0 = float(scipy.special.betaln(pr.a, pr.b))
    elif name == "invgamma":
        pr.family = nat.PRIOR_INVGAMMA
        pr.a = float(shapes[0])
        pr.c0 = float(scipy.special.gammaln(pr.a))
    elif name == "laplace":
        pr.family = nat.PRIOR_LAPLACE
    elif name == "logistic":
        pr.family = nat.PRIOR_LOGISTIC
    elif name == "chi2":
        pr.family = nat.PRIOR_CHI2
        pr.a = float(shapes[0])
        pr.c0 = float(scipy.special.gammaln(pr.a / 2.))
        pr.b = float((numpy.log(2) * pr.a) / 2.)
    else:
        raise ValueError("prior family %r has no device implementation (supported: norm, gamma, uniform, expon, "
                         "halfnorm, lognorm, cauchy, t, beta, invgamma, laplace, logistic, chi2)" % name)
    if not frozen.dist._argcheck(*shapes) or not (float(scale) > 0):
        raise ValueError("invalid parameters for prior %r" % name)
    return pr


WRITER_THREADS = _hostThreads("MCMCN_STORE_THREADS")
# as many as writers: the file's pages are populated while the chains burn in and the writers have nothing to do (C3:
# 37.8 GB in 2.9 s takes eight threads; with four the writers met unpopulated pages and the sampling phase waited)
PREFAULT_THREADS = int(os.environ.get("MCMCN_PREFAULT_THREADS", WRITER_THREADS))


def retainedCount(lo, hi, burn, thin):
    """Number of iterations i in [lo, hi) that Sampler._loop retains (i >= burn and i % thin == 0, :887)."""
    return len(_retainedRange(lo, hi, burn, thin))


class SampleStore(object):
    """Retained samples, device layout [rows][ncol][S] with the chain fastest (include/mcmcn.h), and
    optionally the pointwise log-likelihood of the same rows, [rows][N][S] (saveLogLikelihood).

    resident (``path=None``): every row stays on the device -- ``tensor`` is [nRows][ncol][S].  Tests,
        bench.py and example-scale runs (the CSV writer) use this.
    streamed (``path`` given): the device holds a ring of two chunks of ``chunkRows`` rows.  When the
        chains have filled one chunk it is copied to pinned host memory on a side stream while they
        fill the other, and then written into ``path``, a .npy file [nRows][ncol][nChains] opened with
        numpy.lib.format.open_memmap, by a retire thread (which waits for the copy and deals the rows to
        the writer threads).  The pinned ring mirrors the device ring, one slot per chunk: the thread that
        launches the kernels runs one chunk ahead of the writers and then waits for a slot -- its run-ahead
        being throttled, the device has the next chunk's launches queued meanwhile (4 or 6 slots left the
        sampling loop of config 3 as fast or slower: profiles/experiments/r2_store_pin_slots_ab.log).  Device
        memory is 2 x chunkBytes and pinned memory the same, whatever the run length
        (posteriorSampling.py:898-909, :933-936 appends a CSV row per retained iteration; this is the
        same stream of rows in binary).  ``Engine.run`` splits its iterations at chunk boundaries;
        ``finish()`` drains the ring.
    ``logLikSink(row0, block)`` receives the pointwise log-likelihood rows as host arrays
    [rows][N][nChains] in row order (streamed or not, at ``finish()`` when resident).
    """

    def __init__(self, engine, nRows, dtype=torch.float64, path=None, logLikelihood=False, logLikSink=None,
                 chunkBytes=128 << 20):
        self.engine = engine
        self.nRows = int(nRows)
        self.dtype = dtype
        self.iterations = []
        self._stopPrefault = False
        self.waitedForWriters = 0.0                 # seconds the launching thread stood waiting for a pinned slot
        self.retireWaitedForDevice = 0.0            # seconds the retire thread waited for chunks to leave the device
        self.retireWrote = 0.0                      # seconds it spent writing them into the file
        self.path = path
        self.streamed = path is not None
        self.logLikSink = logLikSink
        dev, S = engine.device, engine.S
        rowBytes = engine.nCol * S * (8 if dtype == torch.float64 else 4)
        if logLikelihood:
            rowBytes += engine.nObservations * S * 8
        if self.streamed:
            self.chunkRows = int(max(1, min(self.nRows, chunkBytes // max(rowBytes, 1))))
            deviceRows = 2 * self.chunkRows
        else:
            self.chunkRows = self.nRows
            deviceRows = self.nRows
        self.tensor = torch.zeros((deviceRows, engine.nCol, S), dtype=dtype, device=dev)
        self.logLik = torch.zeros((deviceRows, engine.nObservations, S), dtype=torch.float64, device=dev) \
            if logLikelihood else None
        self.deviceBytes = self.tensor.numel() * self.tensor.element_size() + \
            (self.logLik.numel() * 8 if self.logLik is not None else 0)
        if self.streamed:
            self._chunk, self._fill, self._done = 0, 0, 0          # ring position; rows already handed to the sink
            self._side = torch.cuda.Stream(dev)
            # The pinned staging buffers (2 x chunkBytes: 0.6 s of cudaHostAlloc at 1 GB) are allocated by a background
            # thread: the first chunk is full only after the burn-in, so the chains start without waiting for them.
            self._pin, self._pinLL = None, None

            def allocatePinned():
                torch.cuda.set_device(dev)                          # the thread's own current device (default: 0)
                pin = [torch.empty((self.chunkRows, engine.nCol, S), dtype=dtype, pin_memory=True)
                       for _ in range(2)]
                pinLL = [torch.empty((self.chunkRows, engine.nObservations, S), dtype=torch.float64, pin_memory=True)
                         for _ in range(2)] if logLikelihood else None
                self._pin, self._pinLL = pin, pinLL
            self._pinThread = threading.Thread(target=allocatePinned, daemon=True)
            self._pinThread.start()
            self._copied = [None, None]                             # per chunk: event of its copy to the pinned slot
            self._written = [None, None]                            # per chunk: future of the retire job reading its slot
            import concurrent.futures
            self._writers = concurrent.futures.ThreadPoolExecutor(max_workers=WRITER_THREADS)
            self._retirer = concurrent.futures.ThreadPoolExecutor(max_workers=1)     # one thread: chunks retire in order
            npdt = numpy.float64 if dtype == torch.float64 else numpy.float32
            self.sink = numpy.lib.format.open_memmap(path, mode="w+", dtype=npdt,
                                                     shape=(self.nRows, engine.nCol, engine.nChains))
            self._prefaulters = [threading.Thread(target=self._prefault, args=(k, PREFAULT_THREADS), daemon=True)
                                 for k in range(PREFAULT_THREADS)]
            for t in self._prefaulters:
                t.start()

    def _prefault(self, k, nThreads):
        """Background thread k of nThreads: have the kernel allocate and map the file's pages (madvise
        MADV_POPULATE_WRITE, Linux >= 5.14; through ctypes, which releases the GIL), 64 MB pieces in file
        order dealt round-robin to the threads, while the chains burn in -- so that the row copies later
        run at memory speed instead of one page fault per 4 KB.  Best effort: stops silently where the
        call is not supported."""
        try:
            libc = ctypes.CDLL(None, use_errno=True)
            page = os.sysconf("SC_PAGE_SIZE")
            addr = self.sink.ctypes.data
            lo = addr - addr % page
            end = addr + self.sink.nbytes
            step = 64 << 20
            lo += k * step
            while lo < end and not self._stopPrefault:
                n = min(step, end - lo)
                if libc.madvise(ctypes.c_void_p(lo), ctypes.c_size_t(n), 23) != 0:     # MADV_POPULATE_WRITE
                    return
                lo += nThreads * step
        except Exception:
            return

    # ---- what Engine.run needs
    def deviceRow(self):
        """Row of ``tensor`` that the next retained iteration goes to, and the capacity limit for this call."""
        if not self.streamed:
            return len(self.iterations), self.nRows
        return self._chunk * self.chunkRows + self._fill, (self._chunk + 1) * self.chunkRows

    def room(self):
        """Retained rows the current call may still produce."""
        if not self.streamed:
            return self.nRows - len(self.iterations)
        return self.chunkRows - self._fill

    def advance(self, iterations):
        """``iterations``: the retained iterations the launches just enqueued will write."""
        self.iterations += iterations
        if not self.streamed:
            return
        self._fill += len(iterations)
        if self._fill == self.chunkRows:
            self._flushChunk()

    # ---- streaming
    def _flushChunk(self):
        c, n = self._chunk, self._fill
        if n == 0:
            return
        if self._pinThread is not None:
            self._pinThread.join()
            self._pinThread = None
            if self._pin is None:
                raise RuntimeError("could not allocate the pinned staging buffers of the sample store")
        if self._written[c] is not None:            # its pinned slot is still being written out: a whole ring behind
            t0 = time.perf_counter()
            self._written[c].result()               # (re-raises what the retire thread raised)
            self.waitedForWriters += time.perf_counter() - t0
        main = torch.cuda.current_stream(self.engine.device)
        filled = torch.cuda.Event()
        filled.record(main)
        self._side.wait_event(filled)
        r0 = c * self.chunkRows
        with torch.cuda.stream(self._side):
            self._pin[c][:n].copy_(self.tensor[r0:r0 + n], non_blocking=True)
            if self.logLik is not None:
                self._pinLL[c][:n].copy_(self.logLik[r0:r0 + n], non_blocking=True)
            done = torch.cuda.Event()
            done.record(self._side)
        self._copied[c] = done
        self._written[c] = self._retirer.submit(self._retire, (c, n, self._done, done))
        self._done += n
        self._chunk, self._fill = 1 - c, 0
        if self._copied[self._chunk] is not None:    # the chains may overwrite the other chunk once it has left the device
            main.wait_event(self._copied[self._chunk])

    def _retire(self, item):
        c, n, row0, copied = item
        t0 = time.perf_counter()
        copied.synchronize()
        t1 = time.perf_counter()
        self.retireWaitedForDevice += t1 - t0
        nC = self.engine.nChains
        src = self._pin[c][:n].numpy()
        # pinned memory -> the file's pages on WRITER_THREADS host threads (numpy copies release the GIL; one
        # thread alone is bound by first-touch page faults of the mapping): whole rows per job when the chunk
        # has many rows, column ranges of a row when it has few
        ncol = src.shape[1]
        perRow = max(1, -(-WRITER_THREADS // n))
        colStep = -(-ncol // perRow)
        jobs = [(r, k0, min(ncol, k0 + colStep)) for r in range(n) for k0 in range(0, ncol, colStep)]

        def put(job):
            r, k0, k1 = job
            self.sink[row0 + r, k0:k1] = src[r, k0:k1, :nC]
        if len(jobs) > 1:
            list(self._writers.map(put, jobs))
        else:
            put(jobs[0])
        if self.logLik is not None and self.logLikSink is not None:
            self.logLikSink(row0, self._pinLL[c][:n].numpy()[:, :, :nC])
        self.retireWrote += time.perf_counter() - t1

    def finish(self):
        """Drain the ring and close the file (streamed), or hand the log-likelihood rows over (resident)."""
        if self.streamed:
            self._flushChunk()
            if self._pinThread is not None:                    # nothing was ever flushed
                self._pinThread.join()
                self._pinThread = None
            for fut in self._written:                          # the last chunks; re-raises a writer's failure
                if fut is not None:
                    fut.result()
            self._retirer.shutdown()
            self._writers.shutdown()
            self._stopPrefault = True
            for t in self._prefaulters:
                t.join()
            self.sink.flush()
        elif self.logLik is not None and self.logLikSink is not None:
            n = len(self.iterations)
            if n:
                self.logLikSink(0, self.logLik[:n, :, :self.engine.nChains].cpu().numpy())

    def hostArray(self):
        """[rows][ncol][nChains] numpy array (the file's memmap when streamed, after finish())."""
        if self.streamed:
            return self.sink[:len(self.iterations)]
        return self.tensor[:len(self.iterations), :, :self.engine.nChains].cpu().numpy()


class Engine(object):
    def __init__(self, objective, nGroups, nResponsesPerGroup, pooling, nChains,
                 priorDistribution=None, chainId0=0, seed=0, device=None, taskObsTarget=256,
                 splitMinObservations=2048):
        if not isinstance(objective, Objective):
            raise TypeError("logLikelihoodFunction must be an Objective handle (device function); "
                            "a Python callable cannot run on the GPU and there is no CPU fallback")
        if pooling not in nat.POOLING_CODE:
            raise Exception("Invalid pooling: ", pooling)
        self.lib = nat.load()
        if not torch.cuda.is_available():
            raise RuntimeError("the MCMC engine needs a CUDA device; there is no CPU fallback")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.objective = objective
        self.pooling = pooling
        self.P = objective.nParameters
        self.nChains = int(nChains)
        self.S = (self.nChains + 31) & ~31
        self.chainId0 = int(chainId0)
        self.seed = int(seed)
        if type(nResponsesPerGroup) == int:
            nResponsesPerGroup = [nResponsesPerGroup] * nGroups
        self.nResponsesPerGroup = [int(r) for r in nResponsesPerGroup]
        self.nObservations = int(sum(self.nResponsesPerGroup))
        if pooling == "complete":                      # :667-671
            self.G = 1
            stepped = [self.nObservations]
        else:
            self.G = int(nGroups)
            stepped = self.nResponsesPerGroup
        if pooling in ("none", "complete"):            # :673-677, :693-697
            if priorDistribution is None or self.P != len(priorDistribution):
                raise ValueError("Invalid prior")
        self.partial = pooling == "partial"
        self.priorScipy = priorDistribution
        self.nCol = self.P * (self.G + (2 if self.partial else 0))
        if self.partial and self.G < 2:
            raise ValueError("partial pooling needs at least 2 groups (the reference divides by nGroups - 1)")

        # ---- model
        # MCMCN_TASK_OBS: observations per task of the FP32-pipe step kernel (a CTA's run of consecutive groups,
        # staged by one TMA copy); results do not depend on it -- a tuning knob for experiments
        taskObsTarget = int(os.environ.get("MCMCN_TASK_OBS", taskObsTarget))
        m, keep = self._buildModel(stepped, pooling, taskObsTarget, tensorCore=True)
        (self._data, self._group_off, self._group_nobs, self._task_group0, self._obj_const, self._tc_data,
         self._tc_group_off, self._group_off_h, self._task_group0_h) = keep
        if not self.partial:
            for p, d in enumerate(priorDistribution):
                m.prior[p] = priorFromScipy(d)
        self.model = m
        if objective.kind != nat.OBJ_USER and not self.lib.mcmcn_supported(
                m.objective, m.n_params, m.n_coef, m.precision):
            raise RuntimeError("objective kind %d with %d parameters (%d coefficients) at %s is not compiled "
                               "into libmcmcn.so" % (m.objective, m.n_params, m.n_coef, objective.precision))

        # ---- chain state
        P, G, S, dev = self.P, self.G, self.S, self.device
        f64 = torch.float64
        self.theta = torch.zeros((P, G, S), dtype=f64, device=dev)
        self.scale = torch.ones((P, G, S), dtype=f64, device=dev)            # :269
        self.counts = torch.zeros((P, G, S), dtype=torch.int32, device=dev)
        self.ll = torch.full((G, S), float("nan"), dtype=f64, device=dev)    # :265
        self.lprior = torch.zeros((P, G, S), dtype=f64, device=dev)
        self.hyper = torch.zeros((5, P, S), dtype=f64, device=dev) if self.partial else None
        self.lpriorStale = False
        st = nat.State()
        st.n_chains = self.nChains
        st.stride = S
        st.chain_id0 = self.chainId0
        st.theta, st.scale, st.counts = _ptr(self.theta), _ptr(self.scale), _ptr(self.counts)
        st.ll, st.lprior, st.hyper = _ptr(self.ll), _ptr(self.lprior), _ptr(self.hyper)
        self.state = st

        # ---- complete pooling at scale: the same observations as groups of 128, evaluated in parallel
        # (mcmcn_model.split); below the threshold one warp per 128 chains steps the single group
        self._split = None
        if pooling == "complete" and self.nObservations >= splitMinObservations:
            N = self.nObservations
            # one accumulator chunk of the tcgen05 evaluation kernel per small group (112 observations for
            # K <= 8, 96 for K = 9..16); every small group centred on the pooled least-squares fit
            size = 128
            if objective.kind == nat.OBJ_LINEAR_REGRESSION and objective.precision == "fp32":
                size = 112 if objective.nCoef <= 8 else 96
            parts = [size] * (N // size) + ([N % size] if N % size else [])
            sm, skeep = self._buildModel(parts, pooling, taskObsTarget, tensorCore=True, commonReference=True)
            scratch = torch.zeros(((P + len(parts) + 3) * S,), dtype=f64, device=dev)
            self._split = (sm, skeep, scratch)
            self.model.split = ctypes.addressof(sm)
            self.model.split_scratch = _ptr(scratch)

    def _buildModel(self, stepped, pooling, taskObsTarget, tensorCore, commonReference=False):
        """Pack the objective's observations as the groups `stepped` and describe them as a
        mcmcn_model (include/mcmcn.h).  Returns the model and the tensors / arrays it points into."""
        objective, dev = self.objective, self.device
        nG = len(stepped)
        data, group_off, group_nobs, obj_const = objective.pack(stepped, commonReference) \
            if commonReference else objective.pack(stepped)
        elem = data.dtype.itemsize
        cap = self.lib.mcmcn_tile_capacity_bytes() // elem
        task_group0 = [0]
        acc_elems, acc_obs = 0, 0
        for g in range(nG):
            e = int(group_off[g + 1] - group_off[g])
            if g > task_group0[-1] and (acc_elems + e > cap or acc_obs + int(group_nobs[g]) > taskObsTarget):
                task_group0.append(g)
                acc_elems, acc_obs = 0, 0
            acc_elems += e
            acc_obs += int(group_nobs[g])
        task_group0.append(nG)
        group_off_h = numpy.ascontiguousarray(group_off, dtype=numpy.int64)
        task_group0_h = numpy.ascontiguousarray(task_group0, dtype=numpy.int32)
        d_data = torch.from_numpy(data).to(dev)
        d_group_off = torch.from_numpy(group_off_h).to(dev)
        d_group_nobs = torch.from_numpy(group_nobs).to(dev)
        d_task_group0 = torch.from_numpy(task_group0_h).to(dev)
        d_obj_const = torch.from_numpy(obj_const).to(dev) if obj_const is not None else None
        tcData = getattr(objective, "tcData", None) if tensorCore else None
        tcOff = getattr(objective, "tcGroupOff", None) if tensorCore else None
        d_tc_data = torch.from_numpy(tcData).to(dev) if tcData is not None else None
        d_tc_group_off = torch.from_numpy(tcOff).to(dev) if tcData is not None else None

        m = nat.Model()
        m.objective = objective.kind
        m.n_params = self.P
        m.n_coef = objective.nCoef
        m.precision = 32 if objective.precision == "fp32" else 64
        m.pooling = nat.POOLING_CODE[pooling]
        m.n_groups = nG
        m.n_tasks = len(task_group0) - 1
        m.n_obj_const = 0 if obj_const is None else len(obj_const)
        m.n_obs = self.nObservations
        m.data = _ptr(d_data)
        m.group_off = _ptr(d_group_off)
        m.group_nobs = _ptr(d_group_nobs)
        m.task_group0 = _ptr(d_task_group0)
        m.task_group0_host = task_group0_h.ctypes.data_as(ctypes.c_void_p)
        m.group_off_host = group_off_h.ctypes.data_as(ctypes.c_void_p)
        m.obj_const = _ptr(d_obj_const)
        m.user_objective = objective.userHandle
        m.tc_data, m.tc_group_off = _ptr(d_tc_data), _ptr(d_tc_group_off)
        m.tc_max_block_floats = int(numpy.diff(tcOff).max()) if tcData is not None else 0
        return m, (d_data, d_group_off, d_group_nobs, d_task_group0, d_obj_const, d_tc_data, d_tc_group_off,
                   group_off_h, task_group0_h)

    # ------------------------------------------------------------------ helpers
    @property
    def usesTensorCore(self):
        """True when mcmcn_run advances this model with the tcgen05 step kernel."""
        return bool(self.lib.mcmcn_uses_tensor_core(ctypes.byref(self.model)))

    @property
    def stepInput(self):
        """The device tensor of observation data the step kernel reads."""
        return self._tc_data if self.usesTensorCore else self._data

    @property
    def stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _up(self, dst, src, lastAxisChains=True):
        """Copy a host array whose last axis is the chain into a [.., S] device tensor."""
        t = torch.from_numpy(numpy.ascontiguousarray(src)).to(self.device)
        dst[..., :self.nChains].copy_(t.to(dst.dtype))

    def _upChainMajor(self, dst, src):
        """Copy a host array whose FIRST axis is the chain ([nC][..]) into a [.., S] device tensor: the
        transposition runs on the device."""
        t = torch.from_numpy(numpy.ascontiguousarray(src)).to(self.device)
        dst[..., :self.nChains].copy_(t.permute(*range(1, t.dim()), 0).to(dst.dtype))

    def setHyper(self, mu, sigma2):
        """mu, sigma2: [P][nChains] host arrays."""
        mu = numpy.asarray(mu, dtype=float)
        sigma2 = numpy.asarray(sigma2, dtype=float)
        with numpy.errstate(all="ignore"):
            sd = numpy.sqrt(sigma2)
            lsd = numpy.log(sd)
            isd = 1.0 / sd
        self._up(self.hyper, numpy.stack([mu, sigma2, sd, lsd, isd]))

    def setState(self, theta, ll, lprior=None, mu=None, sigma2=None, scale=None, counts=None):
        """Host arrays with the chain as LAST axis: theta/lprior/scale [P][G][nC], ll [G][nC]."""
        self._up(self.theta, theta)
        self._up(self.ll, ll)
        if lprior is not None:
            self._up(self.lprior, lprior)
        if scale is not None:
            self._up(self.scale, scale)
        if counts is not None:
            self._up(self.counts, counts)
        if self.partial:
            self.setHyper(mu, sigma2)

    def getState(self):
        n = self.nChains
        out = {"theta": self.theta[..., :n].cpu().numpy(), "ll": self.ll[..., :n].cpu().numpy(),
               "scale": self.scale[..., :n].cpu().numpy(), "lprior": self.lprior[..., :n].cpu().numpy()}
        if self.partial:
            h = self.hyper[..., :n].cpu().numpy()
            out["mu"], out["sigma2"] = h[0], h[1]
        return out

    # ------------------------------------------------------------------ evaluation
    def groupLogLikelihood(self, pooledTheta=None):
        """[G][S] device tensor of group log-likelihoods of the current state, or of
        ``pooledTheta`` ([P][nChains] host array: every group uses the same values)."""
        out = torch.empty((self.G, self.S), dtype=torch.float64, device=self.device)
        pt = None
        if pooledTheta is not None:
            pt = torch.zeros((self.P, self.S), dtype=torch.float64, device=self.device)
            self._up(pt, pooledTheta)
        if self._split is not None and not os.environ.get("MCMCN_NO_SPLIT"):
            # complete pooling at scale: evaluate over the groups of 128 in parallel and add them up in
            # group order (the single stepped group's current values are themselves a pooled vector);
            # the start-state search and the MLE start call this hundreds of times
            sm = self._split[0]
            if pt is None:
                pt = self.theta[:, 0, :].contiguous()
            parts = torch.zeros((sm.n_groups, self.S), dtype=torch.float64, device=self.device)
            nat.call("mcmcn_group_loglik", ctypes.byref(sm), ctypes.byref(self.state), _ptr(pt), _ptr(parts), self.stream)
            nll = torch.zeros((self.S,), dtype=torch.float64, device=self.device)
            nat.call("mcmcn_pooled_nll", int(sm.n_groups), self.S, _ptr(parts), _ptr(nll), self.stream)
            return nll.neg_().reshape(1, self.S)
        nat.call("mcmcn_group_loglik", ctypes.byref(self.model), ctypes.byref(self.state),
                 _ptr(pt), _ptr(out), self.stream)
        return out

    def pooledNll(self, x):
        """MCMC._mleObjectiveFunction (:1102-1105) for every chain: x is [P][nChains]."""
        ll = self.groupLogLikelihood(x)
        out = torch.empty((self.S,), dtype=torch.float64, device=self.device)
        nat.call("mcmcn_pooled_nll", self.G, self.S, _ptr(ll), _ptr(out), self.stream)
        return out[:self.nChains].cpu().numpy()

    def pointwiseLogLikelihood(self):
        """StepMethod.logLikelihood (:656-659): [N][nChains] host array."""
        out = torch.empty((self.nObservations, self.S), dtype=torch.float64, device=self.device)
        nat.call("mcmcn_pointwise_loglik", ctypes.byref(self.model), ctypes.byref(self.state),
                 _ptr(out), self.stream)
        return out[:, :self.nChains].cpu().numpy()

    # ------------------------------------------------------------------ start-up
    def initialise(self, parameterName, startingPointValueRange=None, startWithMLE=False, logger=None):
        """Reference start-up, all chains at once.  Each chain draws from its own legacy
        MT19937 stream seeded with its global chain id (seed = chain, :225, :1015), in the
        reference's order, so start states equal the reference's."""
        from startpoint import findStartingPoints, ChainStreams
        P, G, nC = self.P, self.G, self.nChains
        streams = ChainStreams(nC, self.chainId0)
        x = findStartingPoints(self, streams, parameterName, startingPointValueRange, startWithMLE, logger)
        self.startingPoint = x                                   # [P][nC]

        theta = numpy.zeros((P, G, nC))
        if not self.partial:                                     # :584-592
            lprior = numpy.zeros((P, G, nC))
            for p in range(P):
                theta[p, :, :] = x[p][None, :]
                with numpy.errstate(all="ignore"):
                    lprior[p, :, :] = numpy.asarray(self.priorScipy[p].logpdf(x[p]), dtype=float)[None, :]
            self.setState(theta, numpy.full((G, nC), numpy.nan), lprior)
            return

        # partial pooling, :725-758.  On the host the state is kept chain-major ([nC][P][G]: one chain's draws are
        # contiguous; writing them chain-last cost 4.6 s for 8,192 chains) and transposed on the device.
        mu = x.copy()
        sigma2 = numpy.sqrt(numpy.abs(x) / 10.)                  # sic (:730)
        sd = numpy.sqrt(sigma2)
        muC, sdC = numpy.ascontiguousarray(mu.T)[:, :, None], numpy.ascontiguousarray(sd.T)[:, :, None]   # [nC][P][1]
        # name-major, group-minor: one run of P * G draws per chain is what P calls of G would draw (the stream is sequential)
        z = streams.standardNormal(numpy.arange(nC), P * G).reshape(nC, P, G)
        thetaC = None                                            # host copy of the state: formed only if a group is redrawn
        # numpy.random.normal(mu, sd) = mu + sd * z with two roundings (:740): scaled, shifted and transposed on the device
        # (two separate FP64 kernels, so no fused multiply-add), the normals uploaded as drawn
        zt = torch.from_numpy(z).to(self.device).permute(1, 2, 0)            # [P][G][nC] view
        sdD = torch.from_numpy(sd).to(self.device)[:, None, :]
        muD = torch.from_numpy(mu).to(self.device)[:, None, :]
        self.theta[..., :nC].copy_(torch.add(torch.mul(zt, sdD), muD))
        del zt
        self.ll.fill_(float("nan"))
        self.setHyper(mu, sigma2)
        # The stored log-priors only matter if a group has to be redrawn below (they are then STALE values of the
        # first draw, :284-288; the kernels otherwise recompute the group-level log-prior from mu, sigma2): they
        # are formed when that first happens, from the first draw, not for every run.
        ll = numpy.full((G, nC), numpy.nan)
        for attempt in range(100000):
            cur = self.groupLogLikelihood()[:, :nC].cpu().numpy()
            fin = numpy.isfinite(cur)
            ll[fin] = cur[fin]
            if fin.all():
                break
            if not self.lpriorStale:                             # scipy.stats.norm(mu, sd).logpdf(theta) of the first draw, on the device
                hmu, hsd = self.hyper[0][:, None, :], self.hyper[2][:, None, :]
                y = (self.theta - hmu) / hsd
                lp = -(y * y) / 2.0 - _NORM_PDF_LOGC - torch.log(hsd)
                self.lprior.copy_(torch.where(~(hsd > 0) | torch.isnan(y), torch.full_like(lp, float("nan")), lp))
                del y, lp
            if thetaC is None:                                   # the same values as on the device
                thetaC = z
                thetaC *= sdC
                thetaC += muC
            badT = ~fin.T                                        # [nC][G]
            redo = numpy.nonzero(badT.any(axis=1))[0]
            nBad = badT[redo].sum(axis=1)
            zNew = streams.standardNormal(redo, P * nBad)
            at = 0
            for c, nb in zip(redo, nBad):
                bad = numpy.nonzero(badT[c])[0]
                # name by name, the bad groups in order (:755-758): one run draws what P calls would; log-prior left stale
                thetaC[c][:, bad] = zNew[at:at + P * nb].reshape(P, nb) * sdC[c] + muC[c]
                at += P * nb
            self.lpriorStale = True
            self._upChainMajor(self.theta, thetaC)
        else:
            raise RuntimeError("could not find finite group log-likelihoods for every group")
        self._up(self.ll, ll)

    def collectTiming(self):
        """Wait for the sampled per-kernel events of earlier run(timing=...) calls."""
        nat.call("mcmcn_timing_collect")

    # ------------------------------------------------------------------ run loop
    def run(self, iter0, nIter, burn, thin, store=None, tape=None, trace=False,
            tuneInterval=100, useLpriorOverride=None, timing=None):
        """Advance every chain by nIter iterations (Sampler._loop, :862-896).  With a streamed store the
        iterations are issued in pieces that end where a chunk of the store's ring is full."""
        if store is None or store.room() >= retainedCount(iter0, iter0 + nIter, burn, thin) or tape is not None or trace:
            return self._run(iter0, nIter, burn, thin, store, tape, trace, tuneInterval, useLpriorOverride, timing)
        cur, end = int(iter0), int(iter0 + nIter)
        while cur < end:
            room = store.room()
            if room <= 0:
                raise RuntimeError("sample store is full (%d rows)" % store.nRows)
            # last iteration of this piece = the room-th retained one from `cur` on (or the end of the call)
            kept = _retainedRange(cur, end, burn, thin)
            stop = kept[room - 1] + 1 if len(kept) >= room else end
            self._run(cur, stop - cur, burn, thin, store, None, False, tuneInterval, useLpriorOverride, timing)
            useLpriorOverride = None
            cur = stop
        return None

    def _run(self, iter0, nIter, burn, thin, store, tape, trace, tuneInterval, useLpriorOverride, timing):
        P, G, S = self.P, self.G, self.S
        a = nat.RunArgs()
        a.iter0, a.n_iter, a.burn, a.thin = int(iter0), int(nIter), int(burn), int(thin)
        a.tune_interval = int(tuneInterval)
        a.seed = self.seed
        keep = [tape]
        if tape is not None:
            a.tape_z, a.tape_u = _ptr(tape["z"]), _ptr(tape["u"])
            a.tape_accept = _ptr(tape.get("accept"))
            a.tape_zmu, a.tape_qsig = _ptr(tape.get("zmu")), _ptr(tape.get("qsig"))
        tr = None
        if trace:
            shape = (nIter, P, G, S)
            tr = {"ll": torch.zeros(shape, dtype=torch.float64, device=self.device),
                  "lp": torch.zeros(shape, dtype=torch.float64, device=self.device),
                  "diff": torch.zeros(shape, dtype=torch.float64, device=self.device),
                  "accept": torch.zeros(shape, dtype=torch.uint8, device=self.device)}
            a.trace_ll, a.trace_lp, a.trace_diff = _ptr(tr["ll"]), _ptr(tr["lp"]), _ptr(tr["diff"])
            a.trace_accept = _ptr(tr["accept"])
        kept = []
        if store is not None:
            a.store = _ptr(store.tensor)
            a.store_dtype = 64 if store.dtype == torch.float64 else 32
            a.store_row0, a.store_rows = store.deviceRow()
            a.loglik_store = _ptr(store.logLik)
            kept = list(_retainedRange(iter0, iter0 + nIter, burn, thin))
        if useLpriorOverride is None:
            useLpriorOverride = self.partial and self.lpriorStale and iter0 == 0
        a.use_lprior_override = 1 if useLpriorOverride else 0
        if timing is not None:      # numpy float64[12], see mcmcn_run_args.timing; read with collectTiming()
            a.timing = timing.ctypes.data_as(ctypes.c_void_p)
        nat.call("mcmcn_run", ctypes.byref(self.model), ctypes.byref(self.state), ctypes.byref(a), self.stream)
        if store is not None:
            store.advance(kept)
        if iter0 == 0 and nIter > 0:
            self.lpriorStale = False
        del keep
        return tr
