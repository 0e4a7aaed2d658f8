"""Objective handles -- what ``logLikelihoodFunction`` becomes on the GPU.

The reference takes a Python callable ``f(list[P][N]) -> sequence[N]`` of pointwise
log-likelihoods (posteriorSampling.py:61-102).  Here the objective is a *device
function*: a handle naming a hand-written CUDA objective from the registry plus the
observation data it closes over, or CUDA source compiled by NVRTC
(``Objective.from_source``).  A plain Python callable is rejected with TypeError by
``samplePosterior``; there is no CPU fallback.

Registry (device code in csrc/mcmcn_device.cuh):
  gaussian_distribution   example/distribution.py:18-24
  linear_regression       example/regression.py:53-67, generalised to K coefficients
  bernoulli_logit         SURVEY.md config C5
"""

import collections

import numpy

import mcmcn_native as nat


def _round4(n):
    return (int(n) + 3) & ~3


# What Objective.pack makes of the observations (include/mcmcn.h, mcmcn_model): ``data`` one block per stepped
# group for the FP32-pipe kernels, ``groupOff`` [G+1] block offsets, ``groupNobs`` [G] observations per group,
# ``objConst`` the objective constants or None, ``tcData`` / ``tcGroupOff`` the tcgen05 operand blocks and their
# offsets (linear regression in FP32 with K <= 16; None otherwise).
Packed = collections.namedtuple("Packed", "data groupOff groupNobs objConst tcData tcGroupOff")


class Objective(object):
    """Observation data + which device objective evaluates it.

    precision: "fp32" (FP32 per-observation math, FP64 group sums and priors; the fast
    path) or "fp64" (everything in FP64; used for replay verification).
    """

    def __init__(self, kind, nParameters, precision="fp32"):
        if precision not in ("fp32", "fp64"):
            raise ValueError("precision must be 'fp32' or 'fp64'")
        self.kind = kind
        self.nParameters = int(nParameters)
        self.precision = precision
        self.nCoef = 0
        self.userHandle = None

    # ------------------------------------------------------------ constructors
    @classmethod
    def linear_regression(cls, X, y, precision="fp32"):
        """ll_i = norm(loc=y_i, scale=sigma).logpdf(X_i . b); parameters (b_0..b_{K-1}, sigma)."""
        X = numpy.ascontiguousarray(X, dtype=numpy.float64)
        y = numpy.ascontiguousarray(y, dtype=numpy.float64)
        if X.ndim != 2 or y.ndim != 1 or X.shape[0] != y.shape[0]:
            raise ValueError("X must be [N][K] and y [N]")
        self = cls(nat.OBJ_LINEAR_REGRESSION, X.shape[1] + 1, precision)
        self.nCoef = X.shape[1]
        self.X, self.y = X, y
        self.nObservations = X.shape[0]
        return self

    @classmethod
    def bernoulli_logit(cls, x, y, precision="fp32"):
        """ll_i = y_i*eta_i - log(1+exp(eta_i)), eta_i = a + b*x_i; parameters (a, b)."""
        x = numpy.ascontiguousarray(x, dtype=numpy.float64)
        y = numpy.ascontiguousarray(y, dtype=numpy.float64)
        if x.ndim != 1 or x.shape != y.shape:
            raise ValueError("x and y must be [N]")
        self = cls(nat.OBJ_BERNOULLI_LOGIT, 2, precision)
        self.x, self.y = x, y
        self.nObservations = x.shape[0]
        return self

    @classmethod
    def gaussian_distribution(cls, mu, sd, nResponsesPerGroup, precision="fp32"):
        """ll_i = sum_j norm(mu[j][g(i)], sd[j]).logpdf(theta_j); mu is [P][G], sd is [P]."""
        mu = numpy.ascontiguousarray(mu, dtype=numpy.float64)
        sd = numpy.ascontiguousarray(sd, dtype=numpy.float64)
        if mu.ndim != 2 or sd.shape != (mu.shape[0],):
            raise ValueError("mu must be [P][G] and sd [P]")
        self = cls(nat.OBJ_GAUSSIAN_DISTRIBUTION, mu.shape[0], precision)
        if type(nResponsesPerGroup) == int:
            nResponsesPerGroup = [nResponsesPerGroup] * mu.shape[1]
        self.mu, self.sd = mu, sd
        self.groupOfObservation = numpy.repeat(numpy.arange(mu.shape[1]), nResponsesPerGroup)
        self.nObservations = int(len(self.groupOfObservation))
        return self

    @classmethod
    def from_source(cls, source, nParameters, records, header=None, precision="fp32"):
        """A user objective compiled by NVRTC (north star (1); C ABI in include/mcmcn.h).

        ``source`` is CUDA C++ defining

            __device__ mcmc_real mcmc_obj_loglik(const mcmc_real* theta, const mcmc_real* obs,
                                                 const mcmc_real* hdr, int obs_index, int group);

        returning the pointwise log-likelihood of one observation given its own group's
        ``nParameters`` values (the reference's contract, posteriorSampling.py:61-102: ll[i] may
        depend only on observation i and its group's parameters).  ``records`` is [N][F]: the
        per-observation values the function reads through ``obs`` (F is padded to a multiple of 4);
        ``header`` is an optional [G][H] array of per-group constants read through ``hdr``.
        ``mcmc_real`` is float ("fp32") or double ("fp64")."""
        import ctypes
        records = numpy.ascontiguousarray(records, dtype=numpy.float64)
        if records.ndim != 2:
            raise ValueError("records must be [N][F]")
        self = cls(nat.OBJ_USER, nParameters, precision)
        self.records = records
        self.header = None if header is None else numpy.ascontiguousarray(header, dtype=numpy.float64)
        self.obsFloats = _round4(records.shape[1])
        self.hdrFloats = 0 if header is None else _round4(self.header.shape[1])
        self.nObservations = records.shape[0]
        self.source = source
        handle = ctypes.c_void_p()
        nat.call("mcmcn_user_objective_compile", source.encode("utf-8"), self.nParameters, self.obsFloats,
                 self.hdrFloats, 32 if precision == "fp32" else 64, ctypes.byref(handle))
        self.userHandle = handle
        return self

    def __del__(self):
        try:
            if getattr(self, "userHandle", None):
                nat.load().mcmcn_user_objective_free(self.userHandle)
                self.userHandle = None
        except Exception:
            pass

    # ------------------------------------------------------------ packing
    @property
    def elementDtype(self):
        return numpy.float32 if self.precision == "fp32" else numpy.float64

    def pack(self, nResponsesPerGroup, commonReference=False):
        """Pack the observation data into one block per *stepped* group (include/mcmcn.h,
        mcmcn_model).  ``nResponsesPerGroup`` is the list the step method uses (a single
        entry under complete pooling, posteriorSampling.py:667-671).
        ``commonReference`` (linear regression): every group is centred on the SAME reference point,
        the least-squares fit over all observations, instead of its own fit -- what complete pooling
        split over observations wants: the chain's one candidate vector then has one centred form for
        every small group.
        Returns a Packed record."""
        nResp = [int(r) for r in nResponsesPerGroup]
        if sum(nResp) != self.nObservations:
            raise ValueError("nResponsesPerGroup sums to %d but the objective holds %d observations"
                             % (sum(nResp), self.nObservations))
        dt = self.elementDtype
        if self.kind == nat.OBJ_USER:
            if self.header is not None and self.header.shape[0] != len(nResp):
                raise ValueError("a per-group header cannot be used with %d stepped groups (complete pooling "
                                 "makes one group of all observations)" % len(nResp))
            F, H = self.obsFloats, self.hdrFloats
            sizes = numpy.array([H + r * F for r in nResp], dtype=numpy.int64)
            group_off = numpy.zeros(len(nResp) + 1, dtype=numpy.int64)
            group_off[1:] = numpy.cumsum(sizes)
            data = numpy.zeros(int(group_off[-1]), dtype=dt)
            start = 0
            for g, r in enumerate(nResp):
                blk = data[group_off[g]:group_off[g + 1]]
                if H:
                    blk[:self.header.shape[1]] = self.header[g]
                rec = blk[H:].reshape(r, F)
                rec[:, :self.records.shape[1]] = self.records[start:start + r]
                start += r
            return Packed(data, group_off, numpy.array(nResp, dtype=numpy.int32), None, None, None)
        if self.kind == nat.OBJ_LINEAR_REGRESSION:
            K, KP = self.nCoef, _round4(self.nCoef)
            unit = 4 * KP + 4
        elif self.kind == nat.OBJ_BERNOULLI_LOGIT:
            unit = 8
        elif self.kind == nat.OBJ_GAUSSIAN_DISTRIBUTION:
            P, PP = self.nParameters, _round4(self.nParameters)
            unit = 4 * PP
        else:
            raise ValueError("objective kind %r cannot be packed here" % (self.kind,))
        nquads = [(r + 3) // 4 for r in nResp]
        group_off = numpy.zeros(len(nResp) + 1, dtype=numpy.int64)
        group_off[1:] = numpy.cumsum(numpy.array(nquads, dtype=numpy.int64) * unit)
        data = numpy.zeros(int(group_off[-1]), dtype=dt)
        start = 0
        if self.kind == nat.OBJ_LINEAR_REGRESSION:
            bbar = numpy.zeros((len(nResp), self.nCoef), dtype=numpy.float64)
            pooledFit = numpy.linalg.lstsq(self.X, self.y, rcond=None)[0] if commonReference else None
        for g, r in enumerate(nResp):
            q = nquads[g]
            blk = data[group_off[g]:group_off[g + 1]].reshape(q, unit)
            rows = slice(start, start + r)
            if self.kind == nat.OBJ_LINEAR_REGRESSION:
                # centre the group on its least-squares fit (FP32 conditioning, see LinReg in
                # csrc/mcmcn_device.cuh): store ne = X.bbar - y, keep bbar in FP64
                Xg, yg = self.X[rows], self.y[rows]
                if pooledFit is not None:
                    bbar[g] = pooledFit
                else:
                    bbar[g] = numpy.linalg.lstsq(Xg, yg, rcond=None)[0] if r > 0 else 0.0
                xs = numpy.zeros((q * 4, KP), dtype=dt)
                xs[:r, :K] = Xg
                ys = numpy.zeros(q * 4, dtype=dt)
                ys[:r] = Xg @ bbar[g] - yg                      # ne = x.bbar - y
                # quad layout [KP][4 obs] (coefficient-major), then [4] ne
                blk[:, :4 * KP] = xs.reshape(q, 4, KP).transpose(0, 2, 1).reshape(q, 4 * KP)
                blk[:, 4 * KP:] = ys.reshape(q, 4)
            elif self.kind == nat.OBJ_BERNOULLI_LOGIT:
                xs = numpy.zeros(q * 4, dtype=dt)
                ys = numpy.zeros(q * 4, dtype=dt)
                xs[:r] = self.x[rows]
                ys[:r] = self.y[rows]
                blk[:, :4] = xs.reshape(q, 4)
                blk[:, 4:] = ys.reshape(q, 4)
            else:
                ms = numpy.zeros((q * 4, PP), dtype=dt)
                ms[:r, :P] = self.mu[:, self.groupOfObservation[rows]].T
                blk[:, :] = ms.reshape(q, 4 * PP)
            start += r
        obj_const = tcData = tcGroupOff = None
        if self.kind == nat.OBJ_LINEAR_REGRESSION:
            obj_const = numpy.ascontiguousarray(bbar.reshape(-1))
            if self.precision == "fp32" and self.nCoef <= 16:
                tcData, tcGroupOff = self._packTensorCore(nResp, bbar)
        if self.kind == nat.OBJ_GAUSSIAN_DISTRIBUTION:
            obj_const = numpy.concatenate([self.sd, numpy.log(self.sd)]).astype(numpy.float64)
        return Packed(data, group_off, numpy.array(nResp, dtype=numpy.int32), obj_const, tcData, tcGroupOff)

    def _packTensorCore(self, nResp, bbar):
        """Operand blocks of the tcgen05 step kernel (include/mcmcn.h, mcmcn_model.tc_data): per group the
        slabs X_hi (one per block of 8 coefficients: one for K <= 8, two for K = 9..16), X_lo (likewise)
        and NE, each [Np][8] in the K-major no-swizzle core-matrix layout, the FP32 values split into
        parts that are exact in TF32 (3xTF32)."""
        def tf32(v):
            bits = numpy.ascontiguousarray(v, dtype=numpy.float32).view(numpy.uint32)
            return ((bits + numpy.uint32(0x1000)) & numpy.uint32(0xFFFFE000)).view(numpy.float32)

        def slab(a):                                    # [Np][8] -> core-matrix order
            return a.reshape(a.shape[0] // 8, 8, 2, 4).transpose(0, 2, 1, 3).reshape(-1)

        K = self.nCoef
        KB = 1 if K <= 8 else 2
        nSlabs = 2 * KB + 1
        npad = [max(16, (r + 15) // 16 * 16) for r in nResp]
        off = numpy.zeros(len(nResp) + 1, dtype=numpy.int64)
        off[1:] = numpy.cumsum(numpy.array(npad, dtype=numpy.int64) * 8 * nSlabs)
        data = numpy.zeros(int(off[-1]), dtype=numpy.float32)
        start = 0
        for g, r in enumerate(nResp):
            n = npad[g]
            Xg, yg = self.X[start:start + r], self.y[start:start + r]
            x = numpy.zeros((n, 8 * KB), dtype=numpy.float32)
            x[:r, :K] = Xg
            ne = numpy.zeros(n, dtype=numpy.float32)
            ne[:r] = Xg @ bbar[g] - yg                  # same FP32 values as the FP32-pipe block
            xhi = tf32(x)
            xlo = tf32(x - xhi)
            nes = numpy.zeros((n, 8), dtype=numpy.float32)
            nes[:, 0] = tf32(ne)
            nes[:, 1] = tf32(ne - nes[:, 0])
            nes[:, 2] = (ne - nes[:, 0]) - nes[:, 1]
            blk = data[off[g]:off[g + 1]]
            for kb in range(KB):
                blk[8 * n * kb:8 * n * (kb + 1)] = slab(xhi[:, 8 * kb:8 * kb + 8])
                blk[8 * n * (KB + kb):8 * n * (KB + kb + 1)] = slab(xlo[:, 8 * kb:8 * kb + 8])
            blk[8 * n * 2 * KB:] = slab(nes)
            start += r
        return data, off

    def __call__(self, *args, **kwargs):
        raise TypeError("an Objective is a device function handle; it cannot be called on the host")
