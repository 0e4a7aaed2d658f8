"""The sample store at scale (SURVEY.md section 8f-1): rows streaming through the device ring into the
binary store, the manifest with its shards, and the diagnostics reading it in slabs -- all against the
resident store / in-memory path on the same Philox streams."""

import json

import numpy
import pytest
import scipy.stats

import parity

pytestmark = pytest.mark.gpu


def _engine(nChains=37, G=6, R=20, K=3, pooling="partial", seed=3):
    from engine import Engine
    obj, names, nResp, ranges = parity.syntheticRegression(G=G, R=R, K=K)
    eng = Engine(parity.deviceObjective(obj, nResp, "fp32"), G, nResp, pooling, nChains, chainId0=11, seed=seed)
    eng.initialise(names, ranges)
    return eng, names, obj


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_streamed_store_equals_resident_store(dtype, tmp_path):
    """Same seed, same start: the rows (and the pointwise log-likelihood rows) that stream through a
    two-chunk ring of 3 rows into a .npy file equal the rows of a store that keeps everything on the
    device; the calls are cut at odd places so that pieces end inside, at and across chunk boundaries."""
    import torch
    from engine import SampleStore
    tdt = torch.float64 if dtype == "float64" else torch.float32
    nIter, burn, thin = 140, 40, 3
    nRows = len([i for i in range(nIter) if i >= burn and i % thin == 0])            # 33 rows = 11 chunks of 3
    got = {}
    for mode in ("resident", "streamed"):
        eng, names, obj = _engine()
        ll = []
        rowBytes = eng.nCol * eng.S * (8 if dtype == "float64" else 4) + eng.nObservations * eng.S * 8
        store = SampleStore(eng, nRows, tdt, path=str(tmp_path / "s.npy") if mode == "streamed" else None,
                            logLikelihood=True, logLikSink=lambda r0, blk: ll.append((r0, blk.copy())),
                            chunkBytes=3 * rowBytes)
        if mode == "streamed":
            assert store.streamed and store.chunkRows == 3 and store.tensor.shape[0] == 6
        for a, b in ((0, 17), (17, 50), (50, 51), (51, 52), (52, 101), (101, 140)):
            eng.run(a, b - a, burn, thin, store=store)
        store.finish()
        assert len(store.iterations) == nRows
        rows = numpy.array(store.hostArray())
        assert [r0 for r0, _ in ll] == sorted(r0 for r0, _ in ll)
        got[mode] = (rows, numpy.concatenate([blk for _, blk in ll]), eng.getState()["theta"], store.iterations)
    for a, b in zip(got["resident"], got["streamed"]):
        numpy.testing.assert_array_equal(a, b)
    onDisk = numpy.load(str(tmp_path / "s.npy"))
    assert onDisk.shape == (nRows, 4 * 8, 37) and onDisk.dtype == numpy.dtype(dtype)
    numpy.testing.assert_array_equal(onDisk, got["resident"][0])
    # the log-likelihood rows are the pointwise log-likelihood of the retained state
    assert got["streamed"][1].shape == (nRows, 120, 37) and numpy.isfinite(got["streamed"][1]).all()


def test_diagnostic_over_several_shard_files_equals_one_array(tmp_path, monkeypatch):
    """One process diagnosing a store of several shard files (a multi-rank run's store, read afterwards): the
    half-chains of every slab are gathered from all the shards, and R-hat, ESS, median and HDI equal those over
    the same draws as one array in memory.  Slabs of 4 of the 6 keys, so that a pinned slot is reused by a
    smaller slab."""
    import posteriorSampling as ps
    import sampleDiagnosis as sd
    rs = numpy.random.RandomState(7)
    rows, nChains, world = 40, 7, 3
    header = ["a_mu", "a_sigma2", "a[000]", "a[001]", "b[000]", "b[001]"]
    full = rs.normal(size=(rows, len(header), nChains)).cumsum(axis=0)       # random walks: R-hat well above 1
    d = str(tmp_path) + "/"
    for r in range(world):
        lo, hi = sd.chainRange(nChains, r, world)
        numpy.save(d + "samples.rank%d.npy" % r, full[:, :, lo:hi])
    ps.writeManifest(d, header, list(range(rows)), nChains, world, "partial", "float64")
    monkeypatch.setattr(sd, "SLAB_BYTES", 4 * (2 * nChains) * (rows // 2) * 8)
    dShards = sd.Diagnostic(d)
    assert len(dShards._source.blocks) == world
    monkeypatch.setattr(sd, "SLAB_BYTES", 1 << 30)
    dOne = sd.Diagnostic(samples=numpy.transpose(full, (2, 0, 1)), keys=header)
    for k in header:
        assert dShards.rhat[k] == dOne.rhat[k] and dShards.effectiveN[k] == dOne.effectiveN[k]
        assert dShards.median[k] == dOne.median[k] and dShards.hdi[k] == dOne.hdi[k]


def test_samplePosterior_binary_store_manifest_and_slabbed_diagnostics(tmp_path, monkeypatch, capsys):
    """samplePosterior forced into the binary store (FP64 by default, several ring chunks): same draws
    as the CSV run (which rounds them to 1e-6 with "%f"); Diagnostic / diagnoseSamples over the memory-mapped
    store in slabs of a few keys give exactly what one slab over the same array in memory gives."""
    import posteriorSampling as ps
    import sampleDiagnosis as sd
    import engine
    from objectives import Objective
    obj, names, nResp, ranges = parity.syntheticRegression(G=5, R=12, K=2)
    handle = Objective.linear_regression(obj.X, obj.y)
    args = (6, 400, 100, names, 5, nResp, "partial", handle)
    kw = dict(saveLogLikelihood=False, startingPointValueRange=ranges, displayProgress=False)
    ps.samplePosterior(*args, str(tmp_path / "csv"), **kw)
    monkeypatch.setattr(ps, "CSV_VALUE_LIMIT", 0)
    realStore = engine.SampleStore
    monkeypatch.setattr(ps, "SampleStore", lambda *a, **k: realStore(*a, **dict(k, chunkBytes=7 * 21 * 32 * 8)))
    ps.samplePosterior(*args, str(tmp_path / "bin"), **kw)
    assert ps.lastRun["store"].chunkRows == 7 and ps.lastRun["store"].streamed
    man = json.load(open(str(tmp_path / "bin/sample/manifest.json")))
    assert man["format"] == "mcmcn-samples-2" and man["dtype"] == "float64" and man["nChains"] == 6
    assert man["shards"] == [{"file": "samples.npy", "chains": [0, 6]}] and len(man["iterations"]) == 100
    keysC, csv, _ = sd.loadSamples(str(tmp_path / "csv/sample/"))
    keysB, binary, chains = sd.loadSamples(str(tmp_path / "bin/sample/"))
    assert keysB == keysC and chains == list(range(6))
    numpy.testing.assert_allclose(binary, csv, rtol=0, atol=5.1e-7)       # the CSV is the same draws at "%f"
    # diagnostics: slabs of 4 keys over the memmap == one slab over the same array in memory
    monkeypatch.setattr(sd, "SLAB_BYTES", 4 * 12 * 50 * 8)
    dSlab = sd.Diagnostic(str(tmp_path / "bin/sample/"))
    monkeypatch.setattr(sd, "SLAB_BYTES", 1 << 30)
    dOne = sd.Diagnostic(samples=binary, keys=keysB)
    for k in keysB:
        assert dSlab.rhat[k] == dOne.rhat[k] and dSlab.effectiveN[k] == dOne.effectiveN[k]
        assert dSlab.median[k] == dOne.median[k] and dSlab.hdi[k] == dOne.hdi[k]
    # diagnoseSamples over the binary store: tiny slabs (Summary: 30 rows per slab) and one big slab write and
    # print exactly the same (the tables' content is pinned by the golden tests on the reference's CSV files)
    files = ("diagnostic/diagnosticAssessment.csv", "diagnostic/diagnosticAssessmentHyperOnly.csv",
             "diagnostic/diagnosticAssessmentIndividual.csv", "sample/summary.csv")
    seen = []
    for slab in (6 * 5 * 30 * 8, 1 << 30):
        monkeypatch.setattr(sd, "SLAB_BYTES", slab)
        capsys.readouterr()
        sd.diagnoseSamples(str(tmp_path / "bin"), nFigures=0)
        seen.append([capsys.readouterr().out] + [open(str(tmp_path / "bin" / f)).read() for f in files])
    assert seen[0] == seen[1]
    assert "b0_mu" in seen[0][2] and "groupMedian,sigma" in seen[0][4] and "Summary of individual parameters." in seen[0][0]
    # ... and agree with the CSV run's tables up to the CSV's own 1e-6 rounding of the draws
    dCsv = sd.Diagnostic(str(tmp_path / "csv/sample/"))
    for k in keysB:
        numpy.testing.assert_allclose(dCsv.rhat[k], dOne.rhat[k], rtol=1e-4)
        numpy.testing.assert_allclose(dCsv.median[k], dOne.median[k], atol=2e-6)


def test_float32_store_is_an_opt_in_recorded_in_the_manifest(tmp_path, monkeypatch):
    import posteriorSampling as ps
    from objectives import Objective
    obj, names, nResp, ranges = parity.syntheticRegression(G=5, R=12, K=2)
    monkeypatch.setattr(ps, "CSV_VALUE_LIMIT", 0)
    monkeypatch.setattr(ps, "STORE_DTYPE", "float32")
    ps.samplePosterior(3, 100, 20, names, 5, nResp, "none", Objective.linear_regression(obj.X, obj.y),
                       str(tmp_path / "o"), saveLogLikelihood=False, startingPointValueRange=ranges,
                       priorDistribution=[scipy.stats.norm(0, 10)] * 2 + [scipy.stats.gamma(2)],
                       displayProgress=False)
    man = json.load(open(str(tmp_path / "o/sample/manifest.json")))
    assert man["dtype"] == "float32" and "float32" in man["note"]
    assert numpy.load(str(tmp_path / "o/sample/samples.npy")).dtype == numpy.float32


def test_convergence_from_store_in_slabs_and_wide_rows(monkeypatch):
    """convergenceFromStore over the device-resident store in slabs of columns == Diagnostic on the same
    draws; and a row of more than 65,535 columns (G > 32 K at P = 2) is written back."""
    import torch
    import sampleDiagnosis as sd
    from engine import Engine, SampleStore
    eng, names, obj = _engine(nChains=20, G=7, R=10, K=2)
    store = SampleStore(eng, 30, torch.float32)
    eng.run(0, 120, 60, 2, store=store)
    monkeypatch.setattr(sd, "SLAB_BYTES", 5 * 40 * 15 * 8)              # 5 columns per slab
    rhat, ess = sd.convergenceFromStore(store.tensor, 30, 20)
    draws = numpy.transpose(store.hostArray(), (2, 0, 1)).astype(numpy.float64)
    d = sd.Diagnostic(samples=draws, keys=["k%02d" % i for i in range(eng.nCol)])
    numpy.testing.assert_array_equal(rhat.cpu().numpy(), [d.rhat["k%02d" % i] for i in range(eng.nCol)])
    numpy.testing.assert_array_equal(ess.cpu().numpy(), [d.effectiveN["k%02d" % i] for i in range(eng.nCol)])
    # wide rows
    G = 33000
    obj, names, nResp, ranges = parity.syntheticLogit(G=G, R=2)
    eng = Engine(parity.deviceObjective(obj, nResp, "fp32"), G, nResp, "partial", 32, seed=1)
    eng.initialise(names, ranges)
    assert eng.nCol == 2 * (G + 2) > 65535
    store = SampleStore(eng, 2, torch.float32)
    eng.run(0, 2, 0, 1, store=store)
    rows = store.hostArray()
    st = eng.getState()
    numpy.testing.assert_array_equal(rows[1, 2:G + 2, :], st["theta"][0].astype(numpy.float32))
    numpy.testing.assert_array_equal(rows[1, G + 4:, :], st["theta"][1].astype(numpy.float32))
