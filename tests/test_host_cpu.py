"""CPU-only tests: the C-ABI library loads and exports every symbol include/mcmcn.h declares,
the ctypes structs mirror the C structs, and the host-side logic (schedule, output format,
data packing, prior mapping, batched Nelder-Mead, start-state search, shard merging over
gloo with world_size 2) behaves like the reference / oracle.  No kernel is launched here."""

import ctypes
import json
import os
import re
import subprocess
import sys

import numpy
import pytest
import scipy.optimize
import scipy.stats

from conftest import GOLDEN, ROOT, PKG, goldenPath, loadGolden, oracleObjectiveFromMeta
from oracle import posterior_oracle as po

import mcmcn_native as nat


def _declared():
    text = open(os.path.join(ROOT, "include", "mcmcn.h")).read()
    return sorted(set(re.findall(r"^\s*(?:int|const char\*)\s+(mcmcn_[a-z0-9_]+)\s*\(", text, re.M)))


def test_library_loads_and_exports_every_declared_symbol():
    lib = nat.load()
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), n
        assert n in nat.PROTOTYPES, "no ctypes prototype for %s" % n
    assert lib.mcmcn_version() == 100
    assert lib.mcmcn_tile_capacity_bytes() == 65536
    assert lib.mcmcn_supported(nat.OBJ_LINEAR_REGRESSION, 9, 8, 32) == 1
    assert lib.mcmcn_supported(nat.OBJ_LINEAR_REGRESSION, 7, 6, 32) == 1
    for K in range(1, 17):                                                     # K = 1..16 are compiled in (mcmcn.h: K <= 16)
        assert lib.mcmcn_supported(nat.OBJ_LINEAR_REGRESSION, K + 1, K, 32) == 1
        assert lib.mcmcn_supported(nat.OBJ_LINEAR_REGRESSION, K + 1, K, 64) == 1
    assert lib.mcmcn_supported(nat.OBJ_LINEAR_REGRESSION, 18, 17, 32) == 0
    for P in range(1, 9):                                                      # Gaussian distribution: 1..8 parameters
        assert lib.mcmcn_supported(nat.OBJ_GAUSSIAN_DISTRIBUTION, P, 0, 32) == 1
        assert lib.mcmcn_supported(nat.OBJ_GAUSSIAN_DISTRIBUTION, P, 0, 64) == 1
    assert lib.mcmcn_supported(nat.OBJ_GAUSSIAN_DISTRIBUTION, 9, 0, 32) == 0


def test_ctypes_structs_mirror_the_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mcmcn.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(mcmcn_prior), sizeof(mcmcn_model), sizeof(mcmcn_state), sizeof(mcmcn_run_args),'
                   'offsetof(mcmcn_model, prior), offsetof(mcmcn_run_args, timing));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = list(map(int, subprocess.check_output([str(exe)]).split()))
    assert got == [ctypes.sizeof(nat.Prior), ctypes.sizeof(nat.Model), ctypes.sizeof(nat.State),
                   ctypes.sizeof(nat.RunArgs), nat.Model.prior.offset, nat.RunArgs.timing.offset]


def test_no_cpu_fallback_and_callable_rejected():
    import torch
    from engine import Engine
    from objectives import Objective
    with pytest.raises(TypeError):
        Engine(lambda p: p, 2, 2, "partial", 1)
    if not torch.cuda.is_available():
        obj = Objective.bernoulli_logit(numpy.zeros(4), numpy.zeros(4))
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            Engine(obj, 2, 2, "partial", 1)
    with pytest.raises(TypeError):
        Objective.bernoulli_logit(numpy.zeros(4), numpy.zeros(4))([[0.0] * 4, [0.0] * 4])


def test_burn_thin_and_retained_iterations_follow_the_reference():
    from engine import burnThin, retainedIterations
    for nIter, nSamples in [(1000, 100), (2000, 1000), (600, 100), (240, 120), (400, 100), (7, 7), (20000, 1000)]:
        assert burnThin(nIter, nSamples) == po.burn_thin(nIter, nSamples)
    assert burnThin(1000, 100) == (500, 5) and burnThin(2000, 1000) == (1000, 1)
    assert retainedIterations(1000, 500, 5) == list(range(500, 1000, 5))
    with pytest.raises(Exception):
        burnThin(5, 10)


@pytest.mark.parametrize("case", ["reg_partial", "dist_none", "reg_complete"])
def test_csv_writer_reproduces_reference_files(case, tmp_path):
    import pandas
    import posteriorSampling as ps
    meta = loadGolden(case)
    ref = goldenPath(case, "sample.1.csv")
    d = pandas.read_csv(ref, float_precision="round_trip")
    G = 1 if meta["pooling"] == "complete" else meta["nGroups"]
    header = ps.sampleHeader(meta["parameterName"], G, meta["pooling"])
    assert header == list(d.columns[2:])
    out = tmp_path / "sample.1.csv"
    ps.writeSampleCsv(str(out), 1, header, list(d["index"]), d[header].to_numpy())
    assert open(ref).read() == out.read_text()


def test_regression_packing_is_the_same_residual():
    from objectives import Objective
    rs = numpy.random.RandomState(0)
    nResp = [5, 1, 8, 4, 3]
    N, K = sum(nResp), 3
    X, y = rs.normal(size=(N, K)), 100 + rs.normal(size=N)
    for prec in ("fp32", "fp64"):
        pk = Objective.linear_regression(X, y, prec).pack(nResp)
        data, off, nobs, bbar = pk.data, pk.groupOff, pk.groupNobs, pk.objConst
        KP, unit = 4, 4 * 4 + 4
        bbar = bbar.reshape(len(nResp), K)
        start = 0
        for g, r in enumerate(nResp):
            b = rs.normal(size=K)
            blk = data[off[g]:off[g + 1]].astype(float).reshape(-1, unit)
            x = blk[:, :4 * KP].reshape(-1, KP, 4)                      # [quad][k][obs]
            ne = blk[:, 4 * KP:]                                         # [quad][obs]
            res = numpy.einsum("qkj,k->qj", x[:, :K, :], b - bbar[g]) + ne
            want = X[start:start + r] @ b - y[start:start + r]
            numpy.testing.assert_allclose(res.reshape(-1)[:r], want, rtol=0, atol=2e-5 if prec == "fp32" else 1e-12)
            assert numpy.all(res.reshape(-1)[r:] == 0)                   # padding contributes nothing
            start += r
        assert list(nobs) == nResp and off[-1] == data.size


def test_split_packing_of_complete_pooling_is_the_same_sum_of_squares():
    """Complete pooling at scale packs the observations twice (Engine: mcmcn_model.split): as the
    one stepped group and as groups of 128.  Both packings must give the same residual sum of
    squares for any coefficient vector (each group is centred on its own least-squares fit)."""
    from objectives import Objective
    rs = numpy.random.RandomState(1)
    N, K = 300, 3
    X, y = rs.normal(size=(N, K)), 50 + rs.normal(size=N)
    obj = Objective.linear_regression(X, y, "fp64")
    b = rs.normal(size=K)
    want = float(numpy.sum((X @ b - y) ** 2))
    for stepped in ([N], [128, 128, 44]):
        pk = obj.pack(stepped)
        data, off, nobs, bbar = pk.data, pk.groupOff, pk.groupNobs, pk.objConst
        bbar = bbar.reshape(len(stepped), K)
        unit, total = 4 * 4 + 4, 0.0
        for g in range(len(stepped)):
            blk = data[off[g]:off[g + 1]].reshape(-1, unit)
            res = numpy.einsum("qkj,k->qj", blk[:, :16].reshape(-1, 4, 4)[:, :K, :], b - bbar[g]) + blk[:, 16:]
            total += float(numpy.sum(res ** 2))
        assert abs(total - want) <= 1e-9 * want
        assert int(nobs.sum()) == N


def test_tensor_core_operand_blocks_are_an_exact_3xtf32_split():
    """mcmcn_model.tc_data (include/mcmcn.h): per group [X_hi | X_lo | NE] in the K-major core-matrix
    layout; every part must be exact in TF32 (13 zero low bits) and the parts must add up to the
    same FP32 values the FP32-pipe block holds, so both step kernels evaluate the same residual."""
    from objectives import Objective
    rs = numpy.random.RandomState(1)
    nResp = [5, 17, 1, 200, 16]
    N, K = sum(nResp), 5
    X, y = rs.normal(size=(N, K)), 300 + rs.normal(size=N)
    obj = Objective.linear_regression(X, y, "fp32")
    pk = obj.pack(nResp)
    bbar, tc, tcOff = pk.objConst, pk.tcData, pk.tcGroupOff
    assert tc.dtype == numpy.float32 and len(tcOff) == len(nResp) + 1
    assert numpy.all((tc.view(numpy.uint32) & 0x1FFF) == 0)              # exact in TF32
    bbar = bbar.reshape(len(nResp), K)
    start = 0
    for g, r in enumerate(nResp):
        n = max(16, (r + 15) // 16 * 16)
        blk = tc[tcOff[g]:tcOff[g + 1]]
        assert blk.size == 24 * n

        def unslab(a):                                                   # core-matrix order -> [n][8]
            return a.reshape(n // 8, 2, 8, 4).transpose(0, 2, 1, 3).reshape(n, 8)
        xhi, xlo, ne = unslab(blk[:8 * n]), unslab(blk[8 * n:16 * n]), unslab(blk[16 * n:])
        x32 = numpy.zeros((n, 8), dtype=numpy.float32)
        x32[:r, :K] = X[start:start + r]
        assert numpy.all(numpy.abs((xhi.astype(float) + xlo) - x32) <= numpy.abs(x32) * 2.0 ** -21)
        ne32 = numpy.zeros(n, dtype=numpy.float32)
        ne32[:r] = X[start:start + r] @ bbar[g] - y[start:start + r]
        assert numpy.array_equal(ne[:, 0].astype(float) + ne[:, 1] + ne[:, 2], ne32.astype(float))   # three parts: exact
        assert numpy.all(ne[:, 3:] == 0) and numpy.all(xhi[r:] == 0) and numpy.all(xhi[:, K:] == 0)
        # element (n, k) of a slab sits at float index (n/8)*64 + (k/4)*32 + (n%8)*4 + (k%4)
        for (i, k) in ((0, 0), (r - 1, K - 1), (9 % n, 4)):
            assert blk[(i // 8) * 64 + (k // 4) * 32 + (i % 8) * 4 + (k % 4)] == xhi[i, k]
        start += r


def test_packing_returns_one_record_and_leaves_the_objective_as_it_was():
    """Objective.pack hands everything it packs back in its record (also the tensor-core operand
    blocks, which exist for linear regression in FP32 with K <= 16 only) and sets nothing on the
    objective, so that packing the same objective twice (complete pooling at scale) cannot mix the
    two results."""
    from objectives import Objective
    rs = numpy.random.RandomState(2)
    N = 300
    x, y = rs.normal(size=N), (rs.uniform(size=N) < 0.5).astype(float)
    cases = [(Objective.linear_regression(rs.normal(size=(N, K)), y, prec), K <= 16 and prec == "fp32")
             for K in (2, 16, 17) for prec in ("fp32", "fp64")]
    cases.append((Objective.bernoulli_logit(x, y), False))
    for obj, hasTc in cases:
        before = dict(vars(obj))
        for pk in (obj.pack([N]), obj.pack([128, 128, 44], commonReference=True)):
            assert vars(obj).keys() == before.keys() and all(vars(obj)[k] is v for k, v in before.items())
            assert (pk.tcData is not None) == hasTc and (pk.tcGroupOff is not None) == hasTc
            if hasTc:
                assert pk.tcGroupOff[-1] == pk.tcData.size and len(pk.tcGroupOff) == len(pk.groupNobs) + 1


def test_prior_mapping():
    from engine import priorFromScipy
    pr = priorFromScipy(scipy.stats.gamma(10))
    assert pr.family == nat.PRIOR_GAMMA and pr.a == 10 and pr.scale == 1 and pr.loc == 0
    assert abs(pr.c0 - float(scipy.special.gammaln(10.0))) == 0
    pr = priorFromScipy(scipy.stats.norm(loc=100, scale=10))
    assert (pr.family, pr.loc, pr.scale, pr.log_scale) == (nat.PRIOR_NORM, 100.0, 10.0, float(numpy.log(10.0)))
    assert priorFromScipy(scipy.stats.uniform(-2, 4)).family == nat.PRIOR_UNIFORM
    pr = priorFromScipy(scipy.stats.t(4, 1, 3))
    assert (pr.family, pr.a, pr.loc, pr.scale) == (nat.PRIOR_T, 4.0, 1.0, 3.0)
    assert pr.c0 == float(numpy.log(scipy.special.poch(2.0, 0.5)) - 0.5 * (numpy.log(4.0) + numpy.log(numpy.pi)))
    pr = priorFromScipy(scipy.stats.beta(2, 3, loc=-30, scale=60))
    assert (pr.family, pr.a, pr.b, pr.c0) == (nat.PRIOR_BETA, 2.0, 3.0, float(scipy.special.betaln(2.0, 3.0)))
    for frozen, fam in ((scipy.stats.lognorm(0.8, scale=2), nat.PRIOR_LOGNORM), (scipy.stats.cauchy(0, 5), nat.PRIOR_CAUCHY),
                        (scipy.stats.invgamma(3), nat.PRIOR_INVGAMMA), (scipy.stats.laplace(), nat.PRIOR_LAPLACE),
                        (scipy.stats.logistic(1, 3), nat.PRIOR_LOGISTIC), (scipy.stats.chi2(4), nat.PRIOR_CHI2)):
        assert priorFromScipy(frozen).family == fam
    with pytest.raises(ValueError):
        priorFromScipy(scipy.stats.weibull_min(2))
    with pytest.raises(ValueError):
        priorFromScipy(scipy.stats.gamma(-1))


def _devicePriorFormula(pr, x):
    """The arithmetic of prior_logpdf (csrc/mcmcn_device.cuh) restated in numpy from the SAME record
    the host hands to the device: checks that the constants priorFromScipy forms (c0, b, log_scale)
    are the ones the device formulas need."""
    inf = numpy.inf
    y = numpy.float64((x - pr.loc) / pr.scale)
    f = pr.family
    if not (pr.scale > 0.0) or numpy.isnan(y):                    # the device function's first line
        return numpy.nan
    with numpy.errstate(all="ignore"):
        if f == nat.PRIOR_NORM:
            return -y * y / 2.0 - 0.9189385332046727 - pr.log_scale
        if f == nat.PRIOR_GAMMA:
            r = -inf if y < 0 else ((pr.a - 1.0) * numpy.log(y) if pr.a != 1.0 else 0.0) - y - pr.c0
        elif f == nat.PRIOR_UNIFORM:
            r = 0.0 if 0.0 <= y <= 1.0 else -inf
        elif f == nat.PRIOR_EXPON:
            r = -y if y >= 0 else -inf
        elif f == nat.PRIOR_HALFNORM:
            r = -0.22579135264472741 - 0.5 * (y * y) if y >= 0 else -inf
        elif f == nat.PRIOR_LOGNORM:
            r = -inf if y <= 0 else -(numpy.log(y) ** 2) / pr.c0 - numpy.log(pr.a * y * 2.5066282746310002)
        elif f == nat.PRIOR_CAUCHY:
            ay = abs(y)
            r = -1.1447298858494002 - (numpy.log1p(ay * ay) if ay < 1 else 2.0 * numpy.log(ay) + numpy.log1p((numpy.float64(1.0) / ay) ** 2))
        elif f == nat.PRIOR_T:
            r = pr.c0 - (pr.a + 1.0) / 2.0 * numpy.log1p(y * y / pr.a)
        elif f == nat.PRIOR_BETA:
            r = -inf if (y < 0 or y > 1) else ((pr.b - 1.0) * numpy.log1p(-y) if pr.b != 1.0 else 0.0) + \
                ((pr.a - 1.0) * numpy.log(y) if pr.a != 1.0 else 0.0) - pr.c0
        elif f == nat.PRIOR_INVGAMMA:
            r = -inf if y <= 0 else -(pr.a + 1.0) * numpy.log(y) - pr.c0 - numpy.float64(1.0) / y
        elif f == nat.PRIOR_LAPLACE:
            r = numpy.log(0.5 * numpy.exp(-abs(y)))
        elif f == nat.PRIOR_LOGISTIC:
            t = -abs(y)
            r = t - 2.0 * numpy.log1p(numpy.exp(t))
        elif f == nat.PRIOR_CHI2:
            h = pr.a / 2.0 - 1.0
            r = -inf if y < 0 else (h * numpy.log(y) if h != 0.0 else 0.0) - y / 2.0 - pr.c0 - pr.b
        else:
            raise ValueError(f)
        return r - pr.log_scale


def test_prior_records_reproduce_scipy_logpdf():
    from engine import priorFromScipy
    frozen = [scipy.stats.norm(1, 3), scipy.stats.gamma(2.5, loc=-1, scale=2), scipy.stats.gamma(1.0), scipy.stats.uniform(-2, 4),
              scipy.stats.expon(-6, 4), scipy.stats.halfnorm(0, 3), scipy.stats.lognorm(0.8, scale=2), scipy.stats.cauchy(0, 5),
              scipy.stats.t(4, 1, 3), scipy.stats.beta(2, 3, loc=-30, scale=60), scipy.stats.beta(1, 1), scipy.stats.invgamma(3, scale=2),
              scipy.stats.laplace(0, 4), scipy.stats.logistic(1, 3), scipy.stats.chi2(4), scipy.stats.chi2(2)]
    xs = [-40.0, -30.0, -7.5, -6.0, -2.0, -1.0, -0.3, 0.0, 0.2, 0.5, 0.99, 1.0, 2.0, 3.7, 25.0, 30.0, 400.0, numpy.inf, -numpy.inf, numpy.nan]
    for d in frozen:
        pr = priorFromScipy(d)
        for x in xs:
            with numpy.errstate(all="ignore"):
                want = float(d.logpdf(x))
            got = float(_devicePriorFormula(pr, x))
            if numpy.isfinite(want):
                assert abs(got - want) <= 1e-12 * max(abs(want), 1.0), (d.dist.name, x, got, want)
            else:
                assert (numpy.isnan(got) and numpy.isnan(want)) or got == want, (d.dist.name, x, got, want)


class _FakeEngine(object):
    """Host stand-in for Engine.pooledNll so that the start-up logic runs without a GPU."""

    def __init__(self, f, P, nChains, prior=None):
        self.f, self.P, self.nChains, self.priorScipy = f, P, nChains, prior

    def pooledNll(self, x):
        return numpy.array([self.f(x[:, c]) for c in range(x.shape[1])])


def test_batched_nelder_mead_equals_scipy():
    from startpoint import nelderMead
    A = numpy.array([[3.0, 0.5, 0.1], [0.5, 2.0, 0.3], [0.1, 0.3, 1.0]])

    def f(v):
        return float((v - 1.5) @ A @ (v - 1.5) + 0.1 * numpy.sum(numpy.cos(3 * v)))

    rs = numpy.random.RandomState(4)
    x0 = rs.uniform(-3, 3, size=(3, 7))
    x0[1, 2] = 0.0                                   # exercises the zero-coordinate simplex rule
    eng = _FakeEngine(f, 3, 7)
    x, fx, ok = nelderMead(eng, x0, numpy.ones(7, dtype=bool))
    for c in range(7):
        res = scipy.optimize.minimize(f, x0[:, c], method="Nelder-Mead")
        numpy.testing.assert_allclose(x[:, c], res.x, rtol=1e-12, atol=1e-12)
        assert ok[c] == res.success


def test_start_point_search_consumes_the_reference_stream():
    from startpoint import findStartingPoints, ChainStreams
    meta = loadGolden("reg_none")
    obj, prior = oracleObjectiveFromMeta(meta)
    names = tuple(meta["parameterName"])

    def nll(v):
        with numpy.errstate(all="ignore"):
            return -numpy.sum(obj([numpy.full(100, t) for t in v]))

    for ranges in (meta["startingPointValueRange"], {"b0": [-1, 1]}):       # second: priors for b1, sigma
        eng = _FakeEngine(nll, 3, 4, prior)
        x = findStartingPoints(eng, ChainStreams(4), names, ranges, False)
        for c in range(4):
            oc = po.OracleChain(c, c, 20, 10, names, 10, 10, "none", obj, prior, False, ranges)
            numpy.testing.assert_array_equal(x[:, c], oc.startingPoint)
    with pytest.raises(ValueError):
        findStartingPoints(_FakeEngine(nll, 3, 1, None), ChainStreams(1), names, {"b0": [0, 1]}, False)


def test_native_chain_streams_equal_numpy_legacy_random_state_bit_for_bit():
    """csrc/mcmcn_streams.cu: stream c = numpy.random.RandomState(seed0 + c) (the reference seeds each chain's
    process with the chain index, posteriorSampling.py:225): uniforms, normals with the cached second value,
    refills of the 624-word block, interleaving, and the hand-over of a stream to numpy and back."""
    from startpoint import ChainStreams
    n, seed0 = 37, 1000
    st = ChainStreams(n, seed0)
    ref = [numpy.random.RandomState(seed0 + c) for c in range(n)]
    low, high = [-2.0, 0.5, 1e-3, -1e6], [3.0, 0.75, 7.0, 1e6]
    u = st.uniform(numpy.arange(n), low, high)
    want = numpy.array([[r.uniform(low=a, high=b) for a, b in zip(low, high)] for r in ref])
    numpy.testing.assert_array_equal(u, want)
    # an odd count leaves a cached normal behind; the next call must return it first
    z = st.standardNormal(numpy.arange(n), 2001).reshape(n, 2001)
    numpy.testing.assert_array_equal(z, numpy.array([r.standard_normal(2001) for r in ref]))
    # a subset with ragged counts, then uniforms again (uniforms do not touch the cached normal)
    some = numpy.array([5, 0, 36, 17])
    counts = numpy.array([3, 0, 700, 1])
    z = st.standardNormal(some, counts)
    numpy.testing.assert_array_equal(z, numpy.concatenate([ref[c].standard_normal(k) for c, k in zip(some, counts)]))
    u = st.uniform(some, [0.0], [1.0])[:, 0]
    numpy.testing.assert_array_equal(u, numpy.array([ref[c].uniform(low=0.0, high=1.0) for c in some]))
    # hand a stream to numpy / scipy and take it back
    import scipy.stats
    rs = st.randomState(17)
    got = scipy.stats.gamma(2.5, scale=3.0).rvs(size=5, random_state=rs)
    numpy.testing.assert_array_equal(got, scipy.stats.gamma(2.5, scale=3.0).rvs(size=5, random_state=ref[17]))
    st.adopt(17, rs)
    z = st.standardNormal(numpy.arange(n), 11).reshape(n, 11)
    numpy.testing.assert_array_equal(z, numpy.array([r.standard_normal(11) for r in ref]))
    # seeds beyond 32 bits are refused, like numpy.random.seed
    with pytest.raises(RuntimeError):
        ChainStreams(2, 2 ** 32 - 1)


def _gloo_worker(rank, world, port, tmp):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, PKG)
    import sampleDiagnosis as sd
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rs = numpy.random.RandomState(11)
    x = rs.normal(size=(5, 14, 40))                       # [keys][m][n], all chains
    lo, hi = sd.chainRange(7, rank, world)                # 7 chains = 14 half-chains: 3 on rank 0, 4 on rank 1 (ragged)
    mine = x[:, 2 * lo:2 * hi, :]
    mean = torch.from_numpy(mine.mean(axis=2))
    var = torch.from_numpy(mine.var(axis=2, ddof=1))
    vario = torch.from_numpy(numpy.stack(
        [[((mine[k, :, t:] - mine[k, :, :40 - t]) ** 2).sum() for t in range(40)] for k in range(5)]))
    gm, gv, gvario = sd.mergeShards(mean, var, vario, dist.group.WORLD)
    numpy.save(os.path.join(tmp, "merged.%d.npy" % rank),
               numpy.concatenate([gm.numpy().ravel(), gv.numpy().ravel(), gvario.numpy().ravel()]))
    # key-partitioned exchange of the pooled draws (median / HDI across ranks)
    pooled = torch.from_numpy(numpy.ascontiguousarray(mine.reshape(5, -1)))
    owned = sd.exchangeByKey(pooled, dist.group.WORLD)
    numpy.save(os.path.join(tmp, "owned.%d.npy" % rank), owned.numpy())
    # Summary's exchange: per-(chain, row) values gathered along the chain axis, chain order
    perChain = torch.from_numpy(numpy.ascontiguousarray(x[0, 2 * lo:2 * hi:2, :]))       # [chains of this rank][40]
    numpy.save(os.path.join(tmp, "chains.%d.npy" % rank), sd.gatherChains(perChain, dist.group.WORLD).numpy())
    dist.destroy_process_group()


def test_shard_merge_over_gloo_world_size_2(tmp_path):
    """N > 1 path on CPU: two ranks each hold half of the chains; after the exchange both hold
    the moments of all half-chains in chain order and identical per-lag sums."""
    import torch.multiprocessing as mp
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    a = numpy.load(tmp_path / "merged.0.npy")
    b = numpy.load(tmp_path / "merged.1.npy")
    assert numpy.array_equal(a, b)                        # bit-identical on every rank
    rs = numpy.random.RandomState(11)
    x = rs.normal(size=(5, 14, 40))
    mean, var = x.mean(axis=2), x.var(axis=2, ddof=1)
    vario = numpy.stack([[((x[k, :, t:] - x[k, :, :40 - t]) ** 2).sum() for t in range(40)] for k in range(5)])
    numpy.testing.assert_array_equal(a[:70], mean.ravel())
    numpy.testing.assert_array_equal(a[70:140], var.ravel())
    numpy.testing.assert_allclose(a[140:], vario.ravel(), rtol=1e-13)
    # exchangeByKey: rank r owns keys chainRange(5, r, 2) and holds ALL chains' draws of them, chain order
    import sampleDiagnosis as sd
    for r in range(2):
        lo, hi = sd.chainRange(5, r, 2)
        numpy.testing.assert_array_equal(numpy.load(tmp_path / ("owned.%d.npy" % r)), x[lo:hi].reshape(hi - lo, -1))
        numpy.testing.assert_array_equal(numpy.load(tmp_path / ("chains.%d.npy" % r)), x[0, 0::2, :])


def test_chain_ranges_partition_the_chains():
    import sampleDiagnosis as sd
    for n, w in [(16384, 8), (1024, 3), (7, 2), (8, 8)]:
        cover = []
        for r in range(w):
            lo, hi = sd.chainRange(n, r, w)
            cover += list(range(lo, hi))
        assert cover == list(range(n))


def test_retained_count_matches_the_loop_condition():
    """engine.retainedCount = number of i in [lo, hi) with i >= burn and i % thin == 0 (posteriorSampling.py:887)."""
    from engine import retainedCount
    rs = numpy.random.RandomState(0)
    for _ in range(300):
        lo, n, burn, thin = int(rs.randint(0, 50)), int(rs.randint(0, 60)), int(rs.randint(0, 70)), int(rs.randint(1, 9))
        want = len([i for i in range(lo, lo + n) if i >= burn and i % thin == 0])
        assert retainedCount(lo, lo + n, burn, thin) == want


def test_manifest_lists_the_shards_and_samples_load_in_chain_order(tmp_path):
    """The sharded binary store (one .npy per rank + one manifest.json) as the diagnostics open it:
    shard files are memory-mapped, chains come back in global order; a single-file store and the
    round-1 manifest layout still load."""
    import posteriorSampling as ps
    import sampleDiagnosis as sd
    rs = numpy.random.RandomState(5)
    rows, ncol, nChains, world = 6, 4, 7, 3
    full = rs.normal(size=(rows, ncol, nChains))
    d = str(tmp_path) + "/"
    header = ["a_mu", "a_sigma2", "a[000]", "a[001]"]
    for r in range(world):
        lo, hi = sd.chainRange(nChains, r, world)
        numpy.save(d + "samples.rank%d.npy" % r, full[:, :, lo:hi])
    ps.writeManifest(d, header, list(range(10, 22, 2)), nChains, world, "partial", "float64")
    keys, data, chains = sd.loadSamples(d)
    assert keys == header and chains == list(range(nChains))
    numpy.testing.assert_array_equal(data, numpy.transpose(full, (2, 0, 1)))
    for r in range(world):                                    # one shard per rank under torch.distributed
        src = sd.openSamples(d, rank=r, world=world)
        assert src.sharded and src.chains == list(range(*sd.chainRange(nChains, r, world))) and src.nRows == rows
        assert isinstance(src.blocks[0][0], numpy.memmap)
    assert not sd.openSamples(d, rank=0, world=2).sharded     # shard count != world: everybody reads everything
    # single file, and the manifest the first store version wrote
    one = str(tmp_path / "one") + "/"
    os.makedirs(one)
    numpy.save(one + "samples.npy", full)
    ps.writeManifest(one, header, list(range(6)), nChains, 1, "partial", "float64")
    numpy.testing.assert_array_equal(sd.loadSamples(one)[1], numpy.transpose(full, (2, 0, 1)))
    with open(one + "manifest.json", "w") as h:
        json.dump({"file": "samples.npy", "header": header, "iterations": list(range(6)),
                   "chains": list(range(nChains)), "pooling": "partial", "dtype": "float64"}, h)
    assert sd.loadSamples(one)[2] == list(range(nChains))


def test_diagnostic_tables_and_stdout_text_from_given_statistics(capsys):
    """Diagnostic's table / CSV / stdout code on the reference's own numbers (no device needed): the
    per-key statistics are taken from the oracle, the text must equal the reference's files."""
    import sampleDiagnosis as sd
    from oracle.diagnosis_oracle import DiagnosticOracle
    for case in ("reg_partial", "reg_none", "reg_complete"):
        d = os.path.join(GOLDEN, case)
        o = DiagnosticOracle(d)
        o._compute()
        diag = object.__new__(sd.Diagnostic)
        diag._keys, diag._m = list(o.keys), o._m
        diag._rhat, diag._effectiveN, diag._median, diag._hdi = o.rhat, o.effectiveN, o.median, o.hdi
        diag._assessment = diag._summary = None
        diag._done = True
        diag.partiallyPooled, diag.completelyPooled = o.partiallyPooled, o.completelyPooled
        assert diag._getAssessmentString(False) == open(d + "/diagnosticAssessment.csv").read()
        if diag.partiallyPooled:
            assert diag._getAssessmentString(True) == open(d + "/diagnosticAssessmentHyperOnly.csv").read()
        if not diag.completelyPooled:
            assert diag._getSummaryString() == open(d + "/diagnosticAssessmentIndividual.csv").read()
        capsys.readouterr()
        if diag.completelyPooled:
            diag.print(None, False, False)
        if diag.partiallyPooled:
            diag.print(None, False, True)
        if not diag.completelyPooled:
            diag.print(None, True, False)
        assert capsys.readouterr().out in open(d + "/diagnose.stdout.txt").read()
        with pytest.raises(ValueError, match="Not both|no individual|no hyper"):
            diag.print(None, True, True)


def test_fewer_chains_than_ranks_is_refused_on_every_rank_before_any_collective(monkeypatch, tmp_path):
    """samplePosterior under torch.distributed: nChains < world must raise the same error on EVERY rank before
    the first barrier (a rank-local error after it would leave the other ranks waiting forever)."""
    import posteriorSampling as ps
    from objectives import Objective
    handle = Objective.linear_regression(numpy.ones((20, 1)), numpy.zeros(20))
    for rank in range(4):
        monkeypatch.setattr(ps, "_rankWorld", lambda rank=rank: (rank, 4))
        monkeypatch.setattr(ps, "_barrier", lambda world: (_ for _ in ()).throw(AssertionError("collective reached")))
        with pytest.raises(ValueError, match="fewer chains"):
            ps.samplePosterior(3, 10, 5, ("b0", "sigma"), 2, 10, "partial", handle, str(tmp_path / "o"), displayProgress=False)
    assert not os.path.exists(str(tmp_path / "o"))
