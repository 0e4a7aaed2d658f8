"""Drop-in for the reference's ``sampleDiagnosis`` module, computed on the GPU.

Same public names, signatures, files written and text printed as
``/root/reference/sampleDiagnosis.py`` (``diagnoseSamples`` :11-85, ``Diagnostic`` :88-427,
``Summary`` :430-491, ``computeHpdInterval`` :766-776); figures (``Figure`` :494-759) are out
of scope and skipped.  The reductions run as batched FP64 kernels through the C ABI
(include/mcmcn.h, ``mcmcn_diag_*``); the reference's quirks are kept on purpose: ESS sums
rho from lag 0, the truncation scan tests only even lags, the HDI gap uses Python's
banker's rounding, pooling mode is detected by substring, names are cut to 40 bytes.

Input is either the reference-format ``sample/sample.<chain>.csv`` files or the binary
store (``sample/manifest.json`` + ``samples.npy``) that ``samplePosterior`` writes at scale.
Under ``torch.distributed`` (one process per GPU, chains sharded) the per-half-chain moments
and per-lag sums are exchanged with one all-gather each and merged in rank order.
"""

import ctypes
import glob
import json
import os

import numpy
import pandas
import torch

import mcmcn_native as nat
from mcmcn_native import _hostThreads, _ptr, _rankWorld, chainRange


def _device():
    if not torch.cuda.is_available():
        raise RuntimeError("sampleDiagnosis needs a CUDA device; there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _sortedMedianHdiDevice(x, hdi_p):
    """x: device double [n_keys][len] (destroyed: sorted in place).  Returns device [n_keys][3]
    = median, HDI lower, HDI upper (computeHpdInterval, :766-776)."""
    dev = x.device
    nKeys, length = x.shape
    prob = hdi_p / 100.
    gap = max(1, min(length - 1, round(length * prob)))          # Python banker's rounding
    out = torch.empty((nKeys, 3), dtype=torch.float64, device=dev)
    if nKeys:
        nat.call("mcmcn_diag_sort_keys", _ptr(x), nKeys, length, _stream(dev))
        nat.call("mcmcn_diag_median_hdi", _ptr(x), nKeys, length, gap, _ptr(out), _stream(dev))
    return out


def _sortedMedianHdi(x, hdi_p):
    return _sortedMedianHdiDevice(x, hdi_p).cpu().numpy()


def _rankLengths(length, group, device):
    """Every rank's ``length`` (an int), in rank order: one all-gather."""
    import torch.distributed as dist
    lens = [torch.zeros(1, dtype=torch.int64, device=device) for _ in range(dist.get_world_size(group))]
    dist.all_gather(lens, torch.tensor([length], dtype=torch.int64, device=device), group=group)
    return [int(v) for v in lens]


def exchangeByKey(local, group):
    """Key-partitioned exchange for the pooled order statistics (SURVEY.md section 8e / 8f-3):
    ``local`` is this rank's [n_keys][len_r] draws (len_r may differ between ranks); rank r becomes the
    owner of keys chainRange(n_keys, r) and receives every rank's draws of those keys, concatenated in rank
    (= chain) order: returns [keys_owned][sum of len_r].  One all-to-all over NVLink with NCCL; backends
    without all-to-all (gloo, used by the CPU tests) run the same exchange as one gather per owner."""
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    nKeys, length = local.shape
    lens = _rankLengths(length, group, local.device)
    send = [local[slice(*chainRange(nKeys, r, world))].contiguous() for r in range(world)]
    lo, hi = chainRange(nKeys, rank, world)
    recv = [torch.empty((hi - lo, lens[r]), dtype=local.dtype, device=local.device) for r in range(world)]
    if dist.get_backend(group) == "nccl":
        dist.all_to_all(recv, send, group=group)
    else:
        most = max(lens)                                 # gather wants equal shapes: pad to the longest, trim after
        for r in range(world):
            klo, khi = chainRange(nKeys, r, world)
            padded = torch.zeros((khi - klo, most), dtype=local.dtype, device=local.device)
            padded[:, :length] = send[r]
            got = [torch.empty_like(padded) for _ in range(world)] if r == rank else None
            dist.gather(padded, gather_list=got, dst=dist.get_global_rank(group, r) if group is not None else r,
                        group=group)
            if r == rank:
                recv = [got[q][:, :lens[q]] for q in range(world)]
    return torch.cat(recv, dim=1).contiguous()


def pooledMedianHdi(local, hdi_p, group, keySlab=2048):
    """numpy.median and the HDI (:419-427, :766-776) of every key over ALL ranks' draws without
    any rank ever holding all draws of all keys: keys go through exchangeByKey in slabs, their
    owners sort them, and the [n_keys][3] results are all-gathered.  Returns device [n_keys][3]."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    nKeys = local.shape[0]
    out = torch.empty((nKeys, 3), dtype=torch.float64, device=local.device)
    for k0 in range(0, nKeys, keySlab):
        k1 = min(nKeys, k0 + keySlab)
        mine = _sortedMedianHdiDevice(exchangeByKey(local[k0:k1], group), hdi_p)     # [keys owned in this slab][3]
        owned = [chainRange(k1 - k0, r, world) for r in range(world)]
        pad = torch.zeros((max(hi - lo for lo, hi in owned), 3), dtype=torch.float64, device=local.device)
        pad[:mine.shape[0]] = mine
        parts = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(parts, pad, group=group)
        for (lo, hi), part in zip(owned, parts):
            out[k0 + lo:k0 + hi] = part[:hi - lo]
    return out


def computeHpdInterval(samples, hdi_p=95):
    """sampleDiagnosis.py:766-776."""
    dev = _device()
    x = torch.as_tensor(numpy.ascontiguousarray(samples, dtype=numpy.float64), device=dev).reshape(1, -1).clone()
    res = _sortedMedianHdi(x, hdi_p)
    return (res[0, 1], res[0, 2])


# ------------------------------------------------------------------------------ where the draws come from
SLAB_BYTES = int(os.environ.get("MCMCN_DIAG_SLAB_BYTES", 1 << 30))     # device bytes of half-chains per slab of keys
STAGE_THREADS = _hostThreads("MCMCN_DIAG_THREADS")


class SampleSource(object):
    """The retained draws as the diagnostics want them, without ever materialising more than a slab:
    ``blocks`` is a list of (array [rows][ncol][chains_b], chain ids) in chain order -- numpy arrays,
    numpy memmaps of the binary store's shard files, or device tensors ([rows][ncol][S]: the engine's
    resident store).  ``halfChains(k0, k1)`` gives device double [k1-k0][2 chains][n] for a slab of
    columns (mcmcn_diag_halfchains: every chain's rows split into first / second half, :118-156)."""

    def __init__(self, keys, blocks, nRows):
        self.keys = list(keys)
        self.blocks = blocks                       # [(array-like [rows][ncol][>= chains], [chain ids])]
        self.nRows = int(nRows)
        self.chains = [c for _, ids in blocks for c in ids]
        self.nChains = len(self.chains)
        self._pins, self._pool = {}, None

    @classmethod
    def fromArray(cls, samples, keys, chains=None):
        """samples: [nChains][rows][nKeys] (what loadSamples returns / the CSV files hold)."""
        samples = numpy.asarray(samples, dtype=numpy.float64)
        nC, rows, _ = samples.shape
        block = numpy.ascontiguousarray(numpy.transpose(samples, (1, 2, 0)))       # [rows][keys][chains]
        return cls(keys, [(block, list(chains) if chains is not None else list(range(nC)))], rows)

    @classmethod
    def fromStore(cls, storeTensor, nRows, nChains):
        """The device-resident sample store [rows][ncol][S] (engine.SampleStore.tensor), its first nChains chains."""
        return cls(["c%d" % k for k in range(storeTensor.shape[1])], [(storeTensor, list(range(nChains)))], nRows)

    def stage(self, k0, k1, slot=0):
        """Host half of halfChains: the columns k0..k1 of every host block (numpy array or memmap of a shard
        file) copied into pinned memory, rows split over a few threads (numpy copies release the GIL; one
        thread gathers about 4 GB/s out of a memory-mapped file).  Two slots, so that the next slab can be
        staged while the device works on this one; a slot's buffer is kept while it is large enough (the slabs
        of a pass are all of one size but the last).  Returns one pinned tensor (or None: device block) per block."""
        n = self.nRows // 2
        out = []
        for bi, (arr, ids) in enumerate(self.blocks):
            if isinstance(arr, torch.Tensor):
                out.append(None)
                continue
            nC, nk = len(ids), k1 - k0
            tdt = torch.float64 if arr.dtype == numpy.float64 else torch.float32
            key = (bi, slot)
            pin = self._pins.get(key)
            if pin is None or pin.dtype != tdt or pin.numel() < 2 * n * nk * nC:
                pin = torch.empty((2 * n * nk * nC,), dtype=tdt)
                if torch.cuda.is_available():
                    pin = pin.pin_memory()
                self._pins[key] = pin
            view = pin[:2 * n * nk * nC].view(2 * n, nk, nC)
            dst = view.numpy()
            rowsPer = max(1, -(-2 * n // STAGE_THREADS))
            spans = [(r, min(2 * n, r + rowsPer)) for r in range(0, 2 * n, rowsPer)]

            def copy(span, arr=arr, dst=dst, nC=nC):
                dst[span[0]:span[1]] = arr[span[0]:span[1], k0:k1, :nC]
            if len(spans) > 1:
                list(self._threads().map(copy, spans))
            else:
                copy(spans[0])
            out.append(view)
        return out

    def _threads(self):
        if self._pool is None:
            import concurrent.futures
            self._pool = concurrent.futures.ThreadPoolExecutor(max_workers=STAGE_THREADS)
        return self._pool

    def halfChains(self, k0, k1, dev, staged=None):
        n = self.nRows // 2
        nk = k1 - k0
        out = torch.empty((nk, 2 * self.nChains, n), dtype=torch.float64, device=dev)
        st = _stream(dev)
        if staged is None:
            staged = self.stage(k0, k1)
        j0 = 0
        for (arr, ids), host in zip(self.blocks, staged):
            nC = len(ids)
            if host is None:                                    # resident store: gather straight from it
                src, ncol, stride, kk = arr, arr.shape[1], arr.shape[2], k0
            else:                                               # host rows: this slab of columns only
                src, ncol, stride, kk = host.to(dev, non_blocking=True), nk, nC, 0
            nat.call("mcmcn_diag_halfchains", _ptr(src), 64 if src.dtype == torch.float64 else 32, n, ncol, stride,
                     kk, nk, nC, 2 * self.nChains, j0, _ptr(out), st)
            j0 += 2 * nC
            if host is not None:
                torch.cuda.current_stream(dev).synchronize()    # the pinned slot may be refilled once its copy has left
            del src
        return out

    def columns(self, cols, r0, r1, dev):
        """device double [chains][r1 - r0][len(cols)] (Summary: the groups of one name, rows r0..r1)."""
        parts = []
        for arr, ids in self.blocks:
            nC = len(ids)
            if isinstance(arr, torch.Tensor):
                idx = torch.as_tensor(cols, device=arr.device)
                blk = arr[r0:r1, :, :nC].index_select(1, idx)
            else:
                blk = torch.from_numpy(numpy.ascontiguousarray(arr[r0:r1][:, cols, :nC])).to(dev)
            parts.append(blk.to(torch.float64).permute(2, 0, 1))
        return torch.cat(parts, dim=0).contiguous()


def openSamples(sampleDirectory, rank=0, world=1):
    """SampleSource over what samplePosterior wrote: the binary store when ``manifest.json`` is there
    (shard files are memory-mapped, never read whole), else every ``sample*.csv`` (:102, :132).
    With world > 1 and one shard per rank, rank r opens its own shard only; ``sharded`` says so."""
    manifest = os.path.join(sampleDirectory, "manifest.json")
    if os.path.exists(manifest):
        with open(manifest) as h:
            man = json.load(h)
        shards = man.get("shards") or [{"file": man["file"], "chains": [man["chains"][0], man["chains"][-1] + 1]}]
        sharded = world > 1 and len(shards) == world
        mine = [shards[rank]] if sharded else shards
        blocks = []
        for sh in mine:
            arr = numpy.load(os.path.join(sampleDirectory, sh["file"]), mmap_mode="r")    # [rows][ncol][chains]
            blocks.append((arr, list(range(sh["chains"][0], sh["chains"][1]))))
        src = SampleSource(man["header"], blocks, len(man["iterations"]))
        src.sharded = sharded
        return src
    keys, data, chains = _loadCsv(sampleDirectory)
    src = SampleSource.fromArray(data, keys, chains)
    src.sharded = False
    return src


def _loadCsv(sampleDirectory):
    files = glob.glob(sampleDirectory + "/sample*.csv")
    if not files:
        raise FileNotFoundError("no sample*.csv under %s" % sampleDirectory)

    def chainOf(path):      # sample.<chain>.csv; the reference takes glob order, which is arbitrary
        parts = os.path.basename(path).split(".")
        return int(parts[1]) if len(parts) > 2 and parts[1].isdigit() else 1 << 30

    files.sort(key=lambda f: (chainOf(f), f))
    frames, keys = [], None
    for filename in files:
        d = pandas.read_csv(filename, float_precision="round_trip")
        if keys is None:
            keys = [k for k in d.columns if k not in ("chain", "index")]
        frames.append(d[keys].to_numpy(dtype=numpy.float64))
    return keys, numpy.stack(frames), [chainOf(f) for f in files]


def loadSamples(sampleDirectory):
    """Returns (keys in column order, array [nChains][rows][nKeys] float64, chain ids) -- everything in
    host memory; meant for example-scale runs and tests.  The diagnostics themselves go through
    openSamples / SampleSource and never hold more than a slab."""
    if os.path.exists(os.path.join(sampleDirectory, "manifest.json")):
        src = openSamples(sampleDirectory)
        data = numpy.concatenate([numpy.transpose(numpy.asarray(arr[:, :, :len(ids)], dtype=numpy.float64), (2, 0, 1))
                                  for arr, ids in src.blocks], axis=0)
        return src.keys, numpy.ascontiguousarray(data), src.chains
    return _loadCsv(sampleDirectory)


def gatherShards(t, group):
    """all-gather a [n_keys][m_local][..] tensor along the half-chain axis (dim 1), rank order; ranks may
    hold different numbers of chains (padded to the largest for the collective, trimmed after)."""
    import torch.distributed as dist
    sizes = _rankLengths(t.shape[1], group, t.device)
    most = max(sizes)
    if t.shape[1] < most:
        pad = torch.zeros((t.shape[0], most - t.shape[1]) + tuple(t.shape[2:]), dtype=t.dtype, device=t.device)
        t = torch.cat([t, pad], dim=1)
    parts = [torch.empty_like(t) for _ in sizes]
    dist.all_gather(parts, t.contiguous(), group=group)
    return torch.cat([p[:, :sz] for p, sz in zip(parts, sizes)], dim=1).contiguous()


def mergeShards(mean, var, vario, group):
    """The one exchange the between-chain diagnostics need (SURVEY.md sections 5 and 8e): every
    rank contributes its chains' half-chain means / variances [n_keys][m_local] and its per-lag
    sums [n_keys][n]; returns (mean, var) over all m half-chains and the per-lag sums added in
    fixed rank order, so every rank gets bit-identical results."""
    mean, var = gatherShards(mean, group), gatherShards(var, group)
    parts = gatherShards(vario.reshape(vario.shape[0], 1, vario.shape[1]), group)   # [n_keys][world][n]
    total = torch.zeros_like(vario)
    for r in range(parts.shape[1]):
        total += parts[:, r, :]
    return mean, var, total


def _slabKeys(nKeys, mLocal, n):
    """Keys per slab: SLAB_BYTES of FP64 half-chains, and within the segmented sort's 2^31 items."""
    per = max(1, mLocal * n)
    return int(max(1, min(nKeys, SLAB_BYTES // (8 * per), ((1 << 31) - 1) // per, 65535)))


def _convergenceSlab(x, group, rh):
    """R-hat quadruple of one slab of half-chains x [nk][mLocal][n], written into rh [nk][4]; returns the
    per-lag sums [nk][n] (over all ranks' chains under ``group``) and the number of half-chains m."""
    dev = x.device
    nk, mL, n = x.shape
    st = _stream(dev)
    f64 = torch.float64
    mean = torch.empty((nk, mL), dtype=f64, device=dev)
    var = torch.empty((nk, mL), dtype=f64, device=dev)
    nat.call("mcmcn_diag_moments", _ptr(x), nk, mL, n, _ptr(mean), _ptr(var), st)
    vario = torch.empty((nk, n), dtype=f64, device=dev)
    nat.call("mcmcn_diag_variogram", _ptr(x), nk, mL, n, _ptr(vario), st)
    if group is not None:
        mean, var, vario = mergeShards(mean, var, vario, group)
    m = mean.shape[1]
    nat.call("mcmcn_diag_rhat", _ptr(mean), _ptr(var), nk, m, n, _ptr(rh), st)
    return vario, m


def _slabStatistics(source, dev, group, convergence=False, orderStatistics=False, rho=None, hdi_p=95, timing=None):
    """One pass of the diagnostics over a SampleSource, a slab of keys at a time (_slabKeys); while the device works
    on a slab, a host thread stages the next slab's host rows (sources with host blocks only).  ``convergence``:
    the R-hat quadruple (B, W, vhat, R-hat) and the ESS of every key, and its autocorrelations copied into
    ``rho`` (host [keys][n]) if given; ``orderStatistics``: the median and HDI of every key's pooled draws.
    Under ``group`` (chains sharded over the ranks) ``timing`` receives what this rank exchanged.  Returns device
    (rhat [keys][4], ess [keys], medianHdi [keys][3]), None for what was not asked."""
    import concurrent.futures
    st = _stream(dev)
    f64 = torch.float64
    nKeys, mL, n = len(source.keys), 2 * source.nChains, source.nRows // 2
    rh = torch.empty((nKeys, 4), dtype=f64, device=dev) if convergence else None
    ess = torch.empty((nKeys,), dtype=f64, device=dev) if convergence else None
    mh = torch.empty((nKeys, 3), dtype=f64, device=dev) if orderStatistics else None
    world = 1
    if group is not None:
        import torch.distributed as dist
        world = dist.get_world_size(group)
    step = _slabKeys(nKeys, mL, n)
    slabs = [(k0, min(nKeys, k0 + step)) for k0 in range(0, nKeys, step)]
    ahead = concurrent.futures.ThreadPoolExecutor(max_workers=1) \
        if any(not isinstance(arr, torch.Tensor) for arr, _ in source.blocks) else None

    def stage(i):                                                      # slab i's host rows into pinned slot i & 1
        return ahead.submit(source.stage, *slabs[i], i & 1) if ahead is not None and i < len(slabs) else None
    pending = stage(0)
    gathered = exchanged = 0
    for i, (k0, k1) in enumerate(slabs):
        nk = k1 - k0
        staged = pending.result() if pending is not None else None
        pending = stage(i + 1)                                         # the next slab's rows leave the files meanwhile
        x = source.halfChains(k0, k1, dev, staged)                     # [nk][mL][n]
        r = None
        if convergence:
            vario, m = _convergenceSlab(x, group, rh[k0:k1])
            r = torch.empty((nk, n), dtype=f64, device=dev) if rho is not None else None
            nat.call("mcmcn_diag_ess", _ptr(vario), _ptr(rh[k0:k1]), nk, m, n, _ptr(r), _ptr(ess[k0:k1]), st)
            if group is not None:       # what mergeShards received: all m half-chains' means + variances, every rank's per-lag sums
                gathered += nk * (2 * m + n * world) * 8
        if orderStatistics:
            pooled = x.reshape(nk, mL * n)                             # sorted in place: x is not needed again
            if group is not None:       # key-partitioned all-to-all: no rank holds every key's pooled draws
                mh[k0:k1] = pooledMedianHdi(pooled, hdi_p, group)
                exchanged += pooled.numel() * 8 * (world - 1) // world     # what this rank sent to the other owners
            else:
                mh[k0:k1] = _sortedMedianHdiDevice(pooled, hdi_p)
            del pooled
        if r is not None:
            rho[k0:k1] = r.cpu().numpy()
        del x
    if ahead is not None:
        ahead.shutdown()
    if timing is not None:
        if convergence:
            timing["gathered_bytes"], timing["slabs"] = gathered, len(slabs)
        if orderStatistics:
            timing["exchanged_bytes"] = exchanged
    return rh, ess, mh


def convergenceFromStore(storeTensor, nRows, nChains, group=None, timing=None):
    """R-hat and effective sample size of every column of a device-resident sample store
    ([rows][ncol][S], chain fastest; engine.SampleStore) without leaving the GPU: the same
    kernels and formulas as Diagnostic (:158-255), the rows split into first / second half per
    chain (:118-156), the columns processed in slabs (no transposed copy of the whole store).  With
    ``group`` every rank holds a shard of the chains and the half-chain moments and per-lag sums
    are exchanged by one NCCL all-gather per slab (mergeShards); ``timing`` (a dict) then
    receives the bytes this rank gathered.  Returns (rhat[ncol], ess[ncol]) as device tensors."""
    if int(nRows) // 2 < 2:
        raise ValueError("need at least 4 retained rows per chain")
    rh, ess, _ = _slabStatistics(SampleSource.fromStore(storeTensor, nRows, nChains), storeTensor.device, group,
                                 convergence=True, timing=timing)
    return rh[:, 3].contiguous(), ess


def orderStatisticsFromStore(storeTensor, nRows, nChains, hdi_p=95, group=None, timing=None):
    """numpy.median and the 95 % HDI (:419-427, :766-776) of every column of a device-resident sample
    store, pooled over all chains and rows, in slabs of columns.  With ``group`` the pooled draws of a
    slab go through the key-partitioned all-to-all (pooledMedianHdi): no rank ever holds all draws of all
    columns.  Returns device [ncol][3] = median, HDI lower, HDI upper."""
    return _slabStatistics(SampleSource.fromStore(storeTensor, nRows, nChains), storeTensor.device, group,
                           orderStatistics=True, hdi_p=hdi_p, timing=timing)[2]


def _resolveSource(sampleDirectory, samples, keys, group, source):
    """(SampleSource, process group) of Diagnostic's / Summary's arguments: ``source`` as given, ``samples`` in
    memory, or what openSamples finds under ``sampleDirectory`` -- under torch.distributed with one shard per
    rank each rank opens its own, and the ranks exchange over the world group unless ``group`` is given."""
    if source is None:
        if samples is not None:
            source = SampleSource.fromArray(samples, keys)
        else:
            rank, world = _rankWorld()
            source = openSamples(sampleDirectory, rank, world)
            if source.sharded and group is None:
                import torch.distributed as dist
                group = dist.group.WORLD
    return source, group


class Diagnostic(object):
    def __init__(self, sampleDirectory=None, samples=None, keys=None, group=None, source=None):
        """Diagnostic(sampleDirectory) as in the reference (:89-116).  Alternatively pass
        ``samples`` = array [nChains][rows][nKeys] (+ ``keys``) already in memory, or a SampleSource.
        ``group``: a torch.distributed process group whose ranks each hold a shard of the
        chains; results are then over all ranks' chains."""
        self._source, self._group = _resolveSource(sampleDirectory, samples, keys, group, source)
        self._keys = list(self._source.keys)
        self._organiseSamples()
        self._done = False
        self._hdiP = 95
        self._assessment = None
        self._summary = None

    def _organiseSamples(self):
        """:118-156 -- every chain's rows are split into first / second half (done per slab on the device)."""
        N = self._source.nRows
        n = N // 2
        if N != 2 * n:
            # the reference fails with a broadcast error on an odd row count (SURVEY Q10)
            raise ValueError("could not broadcast input array from shape (%d,) into shape (%d,)" % (N - n, n))
        self._mLocal = 2 * self._source.nChains
        self._n = n
        self.partiallyPooled = any("_" in k for k in self._keys)          # :143-144
        self.completelyPooled = not any("01]" in k for k in self._keys)   # :146-147
        self._m = self._mLocal
        if self._group is not None:
            import torch.distributed as dist
            t = torch.tensor([self._mLocal], dtype=torch.int64, device=_device())
            dist.all_reduce(t, group=self._group)
            self._m = int(t[0])

    # ---------------------------------------------------------------- device pipeline
    def _compute(self):
        if self._done:
            return
        self._rhoArr = numpy.empty((len(self._keys), self._n))
        stats = _slabStatistics(self._source, _device(), self._group, convergence=True, orderStatistics=True,
                                rho=self._rhoArr, hdi_p=self._hdiP)
        rh, ess, mh = (t.cpu().numpy() for t in stats)
        k = self._keys
        self._B = dict(zip(k, rh[:, 0]))
        self._W = dict(zip(k, rh[:, 1]))
        self._vhat = dict(zip(k, rh[:, 2]))
        self._rhat = dict(zip(k, rh[:, 3]))
        self._rho = dict(zip(k, self._rhoArr))
        self._effectiveN = dict(zip(k, ess))
        self._median = dict(zip(k, mh[:, 0]))
        self._hdi = dict((key, (mh[i, 1], mh[i, 2])) for i, key in enumerate(k))
        self._done = True

    @property
    def rhat(self):
        self._compute()
        return self._rhat

    @property
    def effectiveN(self):
        self._compute()
        return self._effectiveN

    @property
    def median(self):
        self._compute()
        return self._median

    @property
    def hdi(self):
        self._compute()
        return self._hdi

    # ---------------------------------------------------------------- tables (:257-405)
    # One column specification per table drives the structured array (what `.assessment` /
    # `.summary` return, as in the reference) and the CSV text; both tables are derived lazily.
    _ASSESSMENT_SPEC = (("parameter", "S40", "'%s'"), ("rhat", float, "%.3f"), ("converged", bool, "%s"),
                        ("effective n", float, "%.3f"), ("enough n", bool, "%s"), ("median", float, "%.3f"),
                        ("HDI lower", float, "%.3f"), ("HDI upper", float, "%.3f"))
    _SUMMARY_SPEC = (("parameter", "S40", "'%s'"), ("rhat min", float, "%.3f"), ("rhat median", float, "%.3f"),
                     ("rhat max", float, "%.3f"), ("proportion converged", float, "%.3f"))

    @staticmethod
    def _structured(spec, records):
        return numpy.array(records, dtype=[(title, kind) for title, kind, _ in spec])

    @staticmethod
    def _csvText(spec, table, keep=None):
        """Header line + one formatted line per record whose (decoded) name passes `keep`."""
        pattern = ",".join(fmt for _, _, fmt in spec)
        lines = [",".join(title for title, _, _ in spec)]
        for record in table:
            label = record["parameter"].decode("ascii")
            if keep is None or keep(label):
                lines.append(pattern % ((label,) + tuple(record)[1:]))
        return "\n".join(lines) + "\n"

    @property
    def assessment(self):
        """Per key: R-hat, converged (< 1.1), ESS, enough (> 10 m), median, HDI; sorted by name bytes (:263-289)."""
        if self._assessment is None:
            self._compute()
            enough = self._m * 10
            records = []
            for key in self._keys:
                rhat, ess = self._rhat[key], self._effectiveN[key]
                lower, upper = self._hdi[key]
                records.append((key.encode(), rhat, rhat < 1.1, ess, ess > enough, self._median[key], lower, upper))
            self._assessment = numpy.sort(self._structured(self._ASSESSMENT_SPEC, records), order="parameter")
        return self._assessment

    def _assess(self):
        return self.assessment

    @property
    def summary(self):
        """Per parameter name, over its per-group keys (those with a '['): min / median / max R-hat and the
        share of converged keys (:297-329)."""
        if self._summary is None:
            perName = {}
            for record in self.assessment:
                label = record["parameter"].decode("ascii")
                if "[" in label:
                    bucket = perName.setdefault(label.split("[")[0], ([], []))
                    bucket[0].append(record["rhat"])
                    bucket[1].append(record["converged"])
            records = [(name, min(r), numpy.median(r), max(r), numpy.mean(c))
                       for name, (r, c) in sorted(perName.items())]
            self._summary = self._structured(self._SUMMARY_SPEC, records)
        return self._summary

    def _summarise(self):
        return self.summary

    def print(self, csvfile, individualSummary, hyperOnly):
        """Write one of the three tables to `csvfile`, or to stdout under its banner when None (:331-379)."""
        refusals = ((individualSummary and self.completelyPooled,
                     "MCMC was completely pooled. There is no individual summary."),
                    (hyperOnly and not self.partiallyPooled,
                     "MCMC was not partially pooled. There is no hyper-parameter."),
                    (individualSummary and hyperOnly, "Choose individualSummary or hyperOnly. Not both."))
        for refused, why in refusals:
            if refused:
                raise ValueError(why)
        text = self._getSummaryString() if individualSummary else self._getAssessmentString(hyperOnly)
        if csvfile is not None:
            with open(csvfile, "w") as h:
                h.write(text)
            return
        banner = "MCMC convergence diagnostic."
        if hyperOnly:
            banner = "MCMC convergence diagnostic for hyper-parameters."
        elif individualSummary:
            banner = "Summary of MCMC convergence diagnostic."
        print(banner)
        _stdout_csv(text)

    def _getAssessmentString(self, hyperOnly):
        keep = (lambda label: "_" in label) if hyperOnly else None       # hyper-parameters: <name>_mu, <name>_sigma2
        return self._csvText(self._ASSESSMENT_SPEC, self.assessment, keep)

    def _getSummaryString(self):
        return self._csvText(self._SUMMARY_SPEC, self.summary)


def gatherChains(v, group):
    """all-gather per-(chain, row) values [chains_r][rows] along the chain axis, rank (= chain) order."""
    return gatherShards(v.unsqueeze(0), group)[0]


class Summary(object):
    """Summarise individual parameter values (:430-491): per (chain, retained row) the mean and the
    median over groups of each parameter name, then mean / median / 95% HDI of those over all chains
    and rows.  The first step is local to a chain, so under ``group`` (chains sharded over ranks) every
    rank reduces its own chains, the per-(chain, row) values are all-gathered in chain order and the
    second step runs on the full vector: the result equals the single-process one bit for bit."""

    def __init__(self, sampleDirectory=None, samples=None, keys=None, group=None, source=None):
        source, group = _resolveSource(sampleDirectory, samples, keys, group, source)
        keys = source.keys
        self._n = source.nRows
        names = sorted(set(name.split("[")[0] for name in keys if "[" in name))
        dev = _device()
        st = _stream(dev)
        nC, nRows = source.nChains, source.nRows
        self._rows = {"groupMean": {}, "groupMedian": {}}
        for name in names:
            cols = [i for i, key in enumerate(keys) if (name + "[") in key]      # substring match, :466-467
            G = len(cols)
            mean = torch.empty((nC, nRows), dtype=torch.float64, device=dev)
            med = torch.empty((nC, nRows), dtype=torch.float64, device=dev)
            # rows in slabs: at most SLAB_BYTES of [chains][rows][G] doubles on the device (and within
            # the segmented sort's 2^31 items)
            step = int(max(1, min(nRows, SLAB_BYTES // max(8 * nC * G, 1), ((1 << 31) - 1) // max(nC * G, 1))))
            for r0 in range(0, nRows, step):
                r1 = min(nRows, r0 + step)
                x = source.columns(cols, r0, r1, dev)                               # [chains][r1-r0][G]
                flat = x.reshape(nC * (r1 - r0), G)
                part = torch.empty((nC * (r1 - r0),), dtype=torch.float64, device=dev)
                nat.call("mcmcn_diag_row_mean", _ptr(flat), flat.shape[0], G, _ptr(part), st)
                mean[:, r0:r1] = part.reshape(nC, r1 - r0)
                if G >= 2:
                    nat.call("mcmcn_diag_sort_keys", _ptr(flat), flat.shape[0], G, st)   # in place: flat is a scratch copy
                    mh3 = torch.empty((flat.shape[0], 3), dtype=torch.float64, device=dev)
                    nat.call("mcmcn_diag_median_hdi", _ptr(flat), flat.shape[0], G, 1, _ptr(mh3), st)
                    med[:, r0:r1] = mh3[:, 0].reshape(nC, r1 - r0)
                else:
                    med[:, r0:r1] = x[:, :, 0]
                del x, flat
            for stat, v in (("groupMean", mean), ("groupMedian", med)):
                if group is not None:
                    v = gatherChains(v, group)
                v = v.reshape(1, -1).contiguous()                                   # chain-major, like the reference's loop
                avg = torch.empty((1,), dtype=torch.float64, device=dev)
                nat.call("mcmcn_diag_row_mean", _ptr(v), 1, v.shape[1], _ptr(avg), st)
                mh = _sortedMedianHdi(v.clone(), 95.)
                self._rows[stat][name] = (float(avg.cpu()[0]), mh[0, 0], mh[0, 1], mh[0, 2])
        self._summarise()

    def _summarise(self):
        lines = ["stats,parameter,mean,median,HDI lower,HDI upper"]
        for stat in ("groupMean", "groupMedian"):
            for name in sorted(self._rows[stat]):
                lines.append("%s,%s,%.4f,%.4f,%.4f,%.4f" % ((stat, name) + self._rows[stat][name]))
        self._summary = "\n".join(lines) + "\n"

    def print(self, csvfile):
        if csvfile is None:
            print("Summary of individual parameters.")
            _stdout_csv(self._summary)
        else:
            with open(csvfile, "w") as h:
                h.write(self._summary)


def diagnoseSamples(outputDirectory, assessConvergence=True, printSummary=True, nFigures=10):
    """Diagnose samples (sampleDiagnosis.py:11-85).  Same files and stdout as the reference; with
    ``nFigures`` > 0 also ``figure/logLikelihood.png``, ``figure/traceplot/traceplot<suffix>.png`` and
    ``figure/bivariate/bivariate<suffix>.png`` for the first nFigures key suffices (:73-85; figures.py
    rasterises them itself).  Under torch.distributed
    with the binary store sharded one file per rank, every rank reduces its own chains (Diagnostic /
    Summary exchange what they must) and rank 0 alone writes and prints."""
    sampleDirectory = outputDirectory + "/sample/"
    diagnosticDirectory = outputDirectory + "/diagnostic/"
    rank, world = _rankWorld()
    speaks = rank == 0
    if speaks:
        os.makedirs(diagnosticDirectory, exist_ok=True)

    if assessConvergence:
        if speaks:
            print("- Convergence Diagnostic -")
        diagnostic = Diagnostic(sampleDirectory)
        diagnostic.assessment                                  # every rank takes part in the exchanges
        pooled, hyper = diagnostic.completelyPooled, diagnostic.partiallyPooled
        # (wanted, file, individualSummary, hyperOnly, echoed to stdout as well)
        reports = ((True, "diagnosticAssessment.csv", False, False, pooled),
                   (hyper, "diagnosticAssessmentHyperOnly.csv", False, True, True),
                   (not pooled, "diagnosticAssessmentIndividual.csv", True, False, True))
        for wanted, fileName, individual, hyperOnly, echo in reports:
            if not (wanted and speaks):
                continue
            diagnostic.print(diagnosticDirectory + "/" + fileName, individual, hyperOnly)
            if echo:
                diagnostic.print(None, individual, hyperOnly)

    if printSummary:
        summary = Summary(sampleDirectory)
        if speaks:
            summary.print(sampleDirectory + "/summary.csv")
            summary.print(None)

    if nFigures > 0 and speaks:                                    # :73-85
        traceplotDirectory = outputDirectory + "/figure/traceplot/"
        bivariateDirectory = outputDirectory + "/figure/bivariate/"
        for directory in (traceplotDirectory, bivariateDirectory):
            os.makedirs(directory, exist_ok=True)
        fig = Figure(sampleDirectory)
        fig.loglikelihood(outputDirectory + "/figure/logLikelihood.png")
        fig.traceplots(traceplotDirectory, nFigures)
        fig.bivariates(bivariateDirectory, nFigures)


def _stdout_csv(content):
    """Tab-indented, comma-spaced echo of a CSV text (:762-763)."""
    print("\t" + "\n\t".join(line.replace(",", ", ") for line in content.split("\n")))


# The reference's ``Figure`` class (sampleDiagnosis.py:494-759): ``loglikelihood``, ``traceplots``, ``traceplot``,
# ``bivariates``, ``bivariate`` with its file names; implemented in figures.py (which imports this module lazily).
from figures import Figure  # noqa: E402,F401
