// mcmcn_device.cuh -- device code of the B200-native MCMC step path (sm_100a).
//
// What the reference does per iteration (posteriorSampling.py:594-613): for each
// parameter name, propose for every group, call the user objective once over
// all observations, sum per group, run the Metropolis decision tree per group,
// tune, then Gibbs-update that name's hyper-parameters.  Here thousands of
// chains advance together:
//
//   * lanes = chains.  A warp holds 32*C chains of ONE group; the group's
//     observation block is staged once into shared memory by a TMA bulk copy
//     and every shared-memory read in the hot loop is a warp-uniform broadcast.
//     Per-group sums are per-thread (no shuffles), FP32 per observation, folded
//     into FP64 every 4 observations (reference: sequential fp64 sum, :631-633).
//   * chain state lives in HBM/L2 as [P][G][S] fp64 arrays (chain fastest) and is
//     touched once per (chain, group, sweep); the hot loop runs from registers.
//   * a sweep over name p needs the hyper-parameters of p from the previous
//     iteration only, so all P sweeps of a group run back to back in one kernel
//     and the P Gibbs updates run in one small kernel per iteration.
//
// This header is also the source NVRTC compiles for user objectives, so it
// includes nothing but mcmcn.h.
#pragma once

#include "mcmcn.h"

namespace mcmcn {

#define MCMCN_LOG_SQRT_2PI 0.91893853320467274178  /* numpy.log(numpy.sqrt(2*numpy.pi)) */

// ---------------------------------------------------------------- small PTX helpers
__device__ __forceinline__ unsigned smem_u32(const void* p) {
    return (unsigned)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(unsigned mb, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mb), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned mb, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
}
// TMA 1-D bulk copy global -> shared, completion signalled on the mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned mb) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(dst), "l"(src), "r"(bytes), "r"(mb) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned mb, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "MCMCN_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra MCMCN_DONE;\n"
        "bra MCMCN_WAIT;\n"
        "MCMCN_DONE:\n"
        "}\n" ::"r"(mb), "r"(parity) : "memory");
}

// ---------------------------------------------------------------- Philox4x32-10
// Counter-based RNG: key = (global chain id, seed), counter = (iteration lo,
// iteration hi | stream kind, name*G+group, attempt).  Independent of launch
// geometry and GPU count (SURVEY.md section 8e).
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}
#define MCMCN_STREAM_SWEEP 0u
#define MCMCN_STREAM_HYPER 1u
#define MCMCN_STREAM_GAMMA 2u

__device__ __forceinline__ uint4 philox_draw(long long chain_id, unsigned long long seed, long long iter,
                                             unsigned kind, unsigned index, unsigned attempt) {
    const uint4 ctr = make_uint4((unsigned)iter, ((unsigned)(iter >> 32) & 0x00FFFFFFu) | (kind << 24), index, attempt);
    const uint2 key = make_uint2((unsigned)chain_id ^ (unsigned)(seed >> 32) * 0x9E3779B1u, (unsigned)seed ^ (unsigned)(chain_id >> 32));
    return philox4x32_10(ctr, key);
}
// log2 of a positive normal float on the MUFU unit (no denormal rescue: the arguments here are
// uniforms >= 2^-33)
__device__ __forceinline__ float lg2_fast(float x) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// standard normal from two 32-bit words (Box-Muller at fp32 resolution, branch-free on the MUFU
// unit: lg2, sqrt, cos; symmetric about 0, |z| <= 5.8)
__device__ __forceinline__ double normal_from(unsigned a, unsigned b) {
    const float u1 = (float)((a >> 8) + 1u) * 5.9604644775390625e-8f;   // (0, 1]
    const float u2 = (float)(b >> 8) * 5.9604644775390625e-8f;          // [0, 1)
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * lg2_fast(u1)));   // -2 ln u1
    return (double)(r * __cosf(6.283185307179586f * u2));
}
// Both Box-Muller branches of the same two words: one Philox call serves two consecutive sweeps
// of the step kernels (the cosine branch the even sweep, the sine branch the odd one).
__device__ __forceinline__ void normal_pair_from(unsigned a, unsigned b, float& zc, float& zs) {
    const float u1 = (float)((a >> 8) + 1u) * 5.9604644775390625e-8f;   // (0, 1]
    const float u2 = (float)(b >> 8) * 5.9604644775390625e-8f;          // [0, 1)
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * lg2_fast(u1)));   // -2 ln u1
    zc = r * __cosf(6.283185307179586f * u2);
    zs = r * __sinf(6.283185307179586f * u2);
}
// (w + 0.5) * 2^-32 in (0, 1) from a 32-bit word without an integer-to-double conversion: the
// word fills the top mantissa bits of a double in [1, 2), then one exact subtraction.
__device__ __forceinline__ double uniform_from32(unsigned w) {
    return __hiloint2double((int)(0x3FF00000u | (w >> 12)), (int)((w << 20) | 0x80000u)) - 1.0;
}
// log(u) < diff decided in FP32 when the margin allows: returns +1 (true), -1 (false) or 0
// (too close to call: the caller falls back to the FP64 logarithm, about once per 10^5
// decisions).  __logf is accurate to 2^-21.41 absolute on [0.5, 2] and 3 ulp elsewhere and
// (float)u adds 6e-8 relative, so |__logf((float)u) - log(u)| < 1e-6 * (1 + |log u|) with a
// wide margin; rounding diff to FP32 moves it by at most 6e-8 relative.
__device__ __forceinline__ int log_u_vs_diff_fast(double u, double diff) {
    const float lu = 0.6931471805599453f * lg2_fast((float)u);
    const float d = (float)diff;
    // one margin for both sides: 2e-6 (1 + |log u|) + 2.4e-7 |diff| covers the errors above and the
    // rounding of the FP32 difference itself
    const float x = d - lu;
    const float m = fmaf(fabsf(d), 2.4e-7f, fmaf(fabsf(lu), 2e-6f, 2e-6f));
    return (x > m) ? 1 : ((x < -m) ? -1 : 0);
}
// uniform in [0,1) with 53 random bits, numpy's recipe (legacy random_sample)
__device__ __forceinline__ double uniform_from(unsigned a, unsigned b) {
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}

// ---------------------------------------------------------------- priors (fp64)
// scipy.stats.norm(loc, scale).logpdf(x): y=(x-loc)/scale; -y**2/2 - log(sqrt(2pi)) - log(scale)
__device__ __forceinline__ double norm_logpdf(double x, double loc, double scale, double log_scale) {
    const double y = __ddiv_rn(__dsub_rn(x, loc), scale);
    const double r = __dsub_rn(__dsub_rn(-0.5 * __dmul_rn(y, y), MCMCN_LOG_SQRT_2PI), log_scale);
    return (!(scale > 0.0) || y != y) ? __longlong_as_double(0x7ff8000000000000LL) : r;
}
// same with the reciprocal of the scale precomputed (group-level prior of partial pooling: two
// evaluations per decision; differs from the quotient form by at most 1 ulp of y).  No validity
// selects: sd = 0 (1/sd = inf, log sd = -inf), sd = nan and x = nan come out as nan through the
// arithmetic itself, x = +-inf and sd = inf as -inf -- what scipy's norm.logpdf returns
// (posteriorSampling.py:293-294, :500-502).
__device__ __forceinline__ double norm_logpdf_inv(double x, double loc, double inv_scale, double log_scale) {
    const double y = __dmul_rn(__dsub_rn(x, loc), inv_scale);
    return __dsub_rn(__dsub_rn(-0.5 * __dmul_rn(y, y), MCMCN_LOG_SQRT_2PI), log_scale);
}
__device__ __forceinline__ bool finite64(double v) {
    return (__double2hiint(v) & 0x7ff00000) != 0x7ff00000;
}
__device__ __forceinline__ void prefetch_l1(const void* p) {
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}
__device__ __forceinline__ double prior_logpdf(const mcmcn_prior& pr, double x) {
    const double ninf = __longlong_as_double(0xfff0000000000000LL);
    const double nan_ = __longlong_as_double(0x7ff8000000000000LL);
    if (pr.family == MCMCN_PRIOR_NORM) return norm_logpdf(x, pr.loc, pr.scale, pr.log_scale);
    const double y = __ddiv_rn(__dsub_rn(x, pr.loc), pr.scale);
    if (!(pr.scale > 0.0) || y != y) return nan_;
    double r;
    switch (pr.family) {
        case MCMCN_PRIOR_GAMMA: {  // xlogy(a-1, y) - y - gammaln(a)
            if (y < 0.0) return ninf;
            const double am1 = pr.a - 1.0;
            const double xl = (am1 == 0.0) ? 0.0 : am1 * log(y);
            r = __dsub_rn(__dsub_rn(xl, y), pr.c0);
            break;
        }
        case MCMCN_PRIOR_UNIFORM:
            if (y < 0.0 || y > 1.0) return ninf;
            r = 0.0;
            break;
        case MCMCN_PRIOR_EXPON:
            if (y < 0.0) return ninf;
            r = -y;
            break;
        case MCMCN_PRIOR_HALFNORM:  // 0.5*log(2/pi) - y*y/2
            if (y < 0.0) return ninf;
            r = __dsub_rn(-0.22579135264472741, 0.5 * __dmul_rn(y, y));
            break;
        case MCMCN_PRIOR_LOGNORM: {  // -log(y)**2 / (2 s**2) - log(s*y*sqrt(2 pi)); y == 0 -> -inf
            if (y <= 0.0) return ninf;
            const double ly = log(y);
            r = __dsub_rn(__ddiv_rn(-__dmul_rn(ly, ly), pr.c0), log(__dmul_rn(__dmul_rn(pr.a, y), 2.5066282746310002)));
            break;
        }
        case MCMCN_PRIOR_CAUCHY: {  // |y| < 1: -log(pi) - log1p(y**2); else -log(pi) - (2 log|y| + log1p((1/|y|)**2))
            const double ay = fabs(y);
            if (ay < 1.0) {
                r = __dsub_rn(-1.1447298858494002, log1p(__dmul_rn(ay, ay)));
            } else {
                const double iy = __ddiv_rn(1.0, ay);
                r = __dsub_rn(-1.1447298858494002, __dadd_rn(__dmul_rn(2.0, log(ay)), log1p(__dmul_rn(iy, iy))));
            }
            break;
        }
        case MCMCN_PRIOR_T:  // c0 - (df + 1)/2 * log1p(y*y/df)
            r = __dsub_rn(pr.c0, __dmul_rn(__ddiv_rn(__dadd_rn(pr.a, 1.0), 2.0), log1p(__ddiv_rn(__dmul_rn(y, y), pr.a))));
            break;
        case MCMCN_PRIOR_BETA: {  // xlog1py(b-1, -y) + xlogy(a-1, y) - betaln(a, b)
            if (y < 0.0 || y > 1.0) return ninf;
            const double bm1 = __dsub_rn(pr.b, 1.0), am1 = __dsub_rn(pr.a, 1.0);
            const double t1 = (bm1 == 0.0) ? 0.0 : __dmul_rn(bm1, log1p(-y));
            const double t2 = (am1 == 0.0) ? 0.0 : __dmul_rn(am1, log(y));
            r = __dsub_rn(__dadd_rn(t1, t2), pr.c0);
            break;
        }
        case MCMCN_PRIOR_INVGAMMA:  // -(a+1) log(y) - gammaln(a) - 1/y; open support in scipy: y == 0 -> -inf
            if (y <= 0.0) return ninf;
            r = __dsub_rn(__dsub_rn(__dmul_rn(-__dadd_rn(pr.a, 1.0), log(y)), pr.c0), __ddiv_rn(1.0, y));
            break;
        case MCMCN_PRIOR_LAPLACE:  // log(0.5 * exp(-|y|)) (scipy has no _logpdf: log of the pdf)
            r = log(__dmul_rn(0.5, exp(-fabs(y))));
            break;
        case MCMCN_PRIOR_LOGISTIC: {  // t = -|y|; t - 2 log1p(exp(t))
            const double t = -fabs(y);
            r = __dsub_rn(t, __dmul_rn(2.0, log1p(exp(t))));
            break;
        }
        case MCMCN_PRIOR_CHI2: {  // xlogy(df/2 - 1, y) - y/2 - gammaln(df/2) - log(2) df / 2
            if (y < 0.0) return ninf;
            const double hm1 = __dsub_rn(__ddiv_rn(pr.a, 2.0), 1.0);
            const double xl = (hm1 == 0.0) ? 0.0 : __dmul_rn(hm1, log(y));
            r = __dsub_rn(__dsub_rn(__dsub_rn(xl, __ddiv_rn(y, 2.0)), pr.c0), pr.b);
            break;
        }
        default:
            return nan_;
    }
    return __dsub_rn(r, pr.log_scale);
}

// ---------------------------------------------------------------- sampler rules
// One copy of each rule of Parameter.step / Parameter.tune, called by every step kernel (sweep_kernel,
// sweep_tc_kernel, the complete-pooling split) so that they cannot drift apart.

// numpy.random.normal(value, sd), posteriorSampling.py:304-306
__device__ __forceinline__ double propose(double cur, double sd, double z) {
    return __dadd_rn(cur, __dmul_rn(sd, z));
}

// The random numbers of sweeps p and p + 1 (p even) of one chain and group: one Philox4x32-10 call at
// counter (p >> 1) * G + g, Box-Muller on words 0-1 (cosine branch: sweep p, sine branch: sweep p + 1),
// words 2 and 3 one accept uniform each (uniform_from32).
struct SweepDraws {
    float z0, z1;
    unsigned u0, u1;
};
__device__ __forceinline__ SweepDraws sweep_draws(long long chain_id, unsigned long long seed, long long iter, int p, int G,
                                                  int g) {
    const uint4 r = philox_draw(chain_id, seed, iter, MCMCN_STREAM_SWEEP, (unsigned)((p >> 1) * G + g), 1u);
    SweepDraws d;
    normal_pair_from(r.x, r.y, d.z0, d.z1);
    d.u0 = r.z;
    d.u1 = r.w;
    return d;
}

// The decision tree of Parameter.step, :334-367, in two parts.  The fast part returns the decision and sets
// `exact` when log(u) against diff is too close to call in FP32 (about once per 10^5 decisions); then
// `decide_exact` settles it with the FP64 logarithm.
__device__ __forceinline__ bool decide_fast(double post_cur, double post_prop, double llp, double diff, double u, bool& exact) {
    const bool b1 = !finite64(post_cur) && finite64(post_prop);
    const bool test = finite64(llp) && finite64(diff);                 // branches 4/5 draw the uniform
    const int fast = log_u_vs_diff_fast(u, diff);
    exact = !b1 && test && fast == 0;
    return b1 || (test && fast > 0);
}
__device__ __forceinline__ bool decide_exact(double u, double diff) { return log(u) < diff; }

// Replay machinery of one iteration: the tapes replace the random numbers (z, u) and the decisions, the
// trace arrays record each decision's inputs.  Null pointers: not in use.
struct StepTapes {
    const double* tape_z;
    const double* tape_u;
    const unsigned char* tape_acc;
    double* tr_ll;
    double* tr_lp;
    double* tr_diff;
    unsigned char* tr_acc;
};
// Records the decision at element `at` when `record`, and returns the taped decision when `force`.
__device__ __forceinline__ bool trace_and_force(const StepTapes& t, size_t at, bool record, bool force, double llp,
                                                double lp_prop, double diff, bool accept) {
    if (record) {
        t.tr_ll[at] = llp;
        t.tr_lp[at] = lp_prop;
        t.tr_diff[at] = diff;
        t.tr_acc[at] = accept ? 1 : 0;
    }
    if (force) accept = t.tape_acc[at] != 0;
    return accept;
}

// Burn-in bookkeeping of one decision: `cnt` packs accepted | rejected << 16 since the last tune; on a tune
// iteration Parameter.tune (:385-437) scales the step size by the acceptance rate and the count restarts.
__device__ __forceinline__ unsigned count_and_tune(unsigned cnt, bool accept, bool tune, double* scale) {
    cnt += accept ? 1u : 0x10000u;
    if (tune) {
        const unsigned na = cnt & 0xFFFFu, nr = cnt >> 16;
        if (na + nr) {
            const double sc = *scale;
            const double rate = (double)na / (double)(na + nr);
            double f = 1.0;
            if (rate < 0.001) f = 0.1;
            else if (rate < 0.05) f = 0.5;
            else if (rate < 0.2) f = 0.9;
            else if (rate > 0.95) f = 10.0;
            else if (rate > 0.75) f = 2.0;
            else if (rate > 0.5) f = 1.1;
            double ns = __dmul_rn(sc, f);
            if (ns == 0.0) ns = sc;
            *scale = ns;
            cnt = 0;
        }
    }
    return cnt;
}

// ---------------------------------------------------------------- objective policies
// A policy restates one reference-style objective as a device function over a group's packed
// block in shared memory.
//   Work<C,T>     the C chains' parameters of the current group in the form the hot loop wants
//   local         FP64 parameter value -> working value
//   accumulate    adds the block's contribution for the C chains at once
//   Aux / aux     per-chain terms of the group log-likelihood outside the observation loop
//   finish        accumulator + Aux -> group log-likelihood
//   pointwise     one observation's log-likelihood (saveLogLikelihood path)

// Where a block handed to `accumulate` sits: group index, index of its first observation within
// the group (non-zero when a large group is streamed in chunks), and the group's header in
// global memory (user objectives).
struct ObsCtx {
    int group;
    int obs0;
    const void* hdr;
};

template <typename T> struct Vec4 {};
template <> struct Vec4<float> {
    __device__ static __forceinline__ void load(const float* p, float (&v)[4]) {
        const float4 t = *reinterpret_cast<const float4*>(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
};
template <> struct Vec4<double> {
    __device__ static __forceinline__ void load(const double* p, double (&v)[4]) {
        const double2 a = *reinterpret_cast<const double2*>(p);
        const double2 b = *reinterpret_cast<const double2*>(p + 2);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    }
};
__device__ __forceinline__ float fma_t(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fma_t(double a, double b, double c) { return fma(a, b, c); }

// Parameters as a plain register array; `p` is a run-time index, `c` is always a literal after
// unrolling, so every access below is a chain of selects, never local memory.
template <int P, int C, typename T>
struct PlainWork {
    T th[C][P];
    __device__ __forceinline__ void set(int c, int p, T v) {
#pragma unroll
        for (int k = 0; k < P; ++k) if (k == p) th[c][k] = v;
    }
    __device__ __forceinline__ T get(int c, int p) const {
        T r = th[c][0];
#pragma unroll
        for (int k = 1; k < P; ++k) if (k == p) r = th[c][k];
        return r;
    }
    __device__ __forceinline__ void row(int c, T (&out)[P]) const {
#pragma unroll
        for (int k = 0; k < P; ++k) out[k] = th[c][k];
    }
};

// Packed FP32x2 FMA (PTX fma.rn.f32x2, SASS FFMA2; new on sm_100).  A 64-bit operand is an
// aligned even/odd register pair, so an FFMA2 with one operand served from the reuse cache
// reads exactly one register per bank per FMA: measured 116.7 FMA lanes/clk/SM on B200 whatever
// registers ptxas picks, against 98.4 for scalar FFMA in the same x*b[c]+r[c] pattern (the second
// and third source collide in the even/odd bank about one time in three) and 124.6 for the
// pipe itself (tools/fma_probe.cu).  It also halves the issue slots the FMAs take.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 ffma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
    return d;
}
__device__ __forceinline__ float lo2(f32x2 v) {
    float lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
    return lo;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fadd2(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
// four consecutive floats (16-byte aligned) as two packed pairs: one 128-bit load, the pairs are its registers
__device__ __forceinline__ void load_pairs(const float* p, f32x2& a, f32x2& b) {
    const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(p);
    a = v.x;
    b = v.y;
}
__device__ __forceinline__ float sum2(f32x2 v) {
    float lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
    return lo + hi;
}

// The per-chain terms of a policy whose group log-likelihood is the accumulator itself (all but LinReg).
struct NoAux {
    struct Aux {};
    static constexpr int AUX_DOUBLES = 0;
    __device__ static __forceinline__ void aux_put(const Aux&, double*, int) {}
    __device__ static __forceinline__ Aux aux_get(const double*, int) { return Aux(); }
    template <int C, typename T, class W>
    __device__ static __forceinline__ Aux aux(int, const W&, int) { return Aux(); }
    __device__ static __forceinline__ bool aux_depends_on(int) { return false; }
    __device__ static __forceinline__ double finish(double acc, const Aux&) { return acc; }
};

// Linear regression with K coefficients and a noise sd (example/regression.py:53-67):
//   ll_i = norm(loc=y_i, scale=sigma).logpdf(x_i . b)
// Block: ceil(R/4) quads of [KP][4 obs] x (coefficient-major, so one 128-bit shared load is
// two observation pairs of one coefficient) followed by [4] ne.  Padding observations are
// all-zero and contribute exactly 0.
// FP32 conditioning: the residual x_i.b - y_i cancels catastrophically when |y| >> |residual|
// (the reference's own example has |y| ~ 300 against residuals ~ 1).  The host therefore
// centres every group on a reference point bbar_g (its least-squares fit, FP64, in
// obj_const[g*K + k]) and stores ne_i = x_i.bbar_g - y_i instead of y_i; the kernel evaluates
// the identical residual as x_i.(b - bbar_g) + ne_i with (b - bbar_g) formed in FP64.
template <int K_>
struct LinReg {
    static constexpr int K = K_;
    static constexpr int P = K_ + 1;
    static constexpr int KP = (K_ + 3) & ~3;
    static constexpr int UNIT = 4 * KP + 4;      // elements per quad
    static constexpr int HDR = 0;
    static constexpr int OBS_PER_UNIT = 4;

    template <typename T>
    __device__ static __forceinline__ T local(int p, double v, const double* cst, int g) {
        return (T)(p < K ? __dsub_rn(v, cst[(size_t)g * K + p]) : v);
    }

    // FP64: plain array.  FP32: every coefficient duplicated into an FFMA2 operand pair.
    template <int C, typename T, int Dummy = 0>
    struct Work : PlainWork<P, C, T> {
        __device__ __forceinline__ double sigma(int c) const { return (double)this->th[c][K]; }
    };
    template <int C, int Dummy>
    struct Work<C, float, Dummy> {
        f32x2 b2[C][K];
        float sg[C];
        __device__ __forceinline__ void set(int c, int p, float v) {
#pragma unroll
            for (int k = 0; k < K; ++k) if (k == p) b2[c][k] = pack2(v, v);
            if (p == K) sg[c] = v;
        }
        __device__ __forceinline__ float get(int c, int p) const {
            float r = sg[c];
#pragma unroll
            for (int k = 0; k < K; ++k) if (k == p) r = lo2(b2[c][k]);
            return r;
        }
        __device__ __forceinline__ void row(int c, float (&out)[P]) const {
#pragma unroll
            for (int k = 0; k < K; ++k) out[k] = lo2(b2[c][k]);
            out[K] = sg[c];
        }
        __device__ __forceinline__ double sigma(int c) const { return (double)sg[c]; }
    };

    // FP32 hot loop: sum of squared residuals of C chains over the block, two observations per
    // FFMA2, FP32 partial sums folded into FP64 every 16 observations.
    template <int C>
    __device__ static __forceinline__ void accumulate(const float* __restrict__ blk, int nobs, const double*,
                                                      const Work<C, float>& w, double (&acc)[C], const ObsCtx&) {
        const int nq = (nobs + 3) >> 2;
        for (int q0 = 0; q0 < nq; q0 += 4) {
            f32x2 s2[C];
#pragma unroll
            for (int c = 0; c < C; ++c) s2[c] = 0ull;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (q0 + u < nq) {
                    const float* xq = blk + (size_t)(q0 + u) * UNIT;
                    const ulonglong2 ne = *reinterpret_cast<const ulonglong2*>(xq + 4 * KP);
                    f32x2 r[C][2];
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(xq + 4 * k);
#pragma unroll
                        for (int c = 0; c < C; ++c) r[c][0] = ffma2(x.x, w.b2[c][k], k == 0 ? ne.x : r[c][0]);
#pragma unroll
                        for (int c = 0; c < C; ++c) r[c][1] = ffma2(x.y, w.b2[c][k], k == 0 ? ne.y : r[c][1]);
                    }
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        s2[c] = ffma2(r[c][0], r[c][0], s2[c]);
                        s2[c] = ffma2(r[c][1], r[c][1], s2[c]);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < C; ++c) acc[c] += (double)sum2(s2[c]);
        }
    }
    // FP64 path (replay verification): same layout, scalar FMAs.
    template <int C>
    __device__ static __forceinline__ void accumulate(const double* __restrict__ blk, int nobs, const double*,
                                                      const Work<C, double>& w, double (&acc)[C], const ObsCtx&) {
        const int nq = (nobs + 3) >> 2;
        for (int q = 0; q < nq; ++q) {
            const double* xq = blk + (size_t)q * UNIT;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    double r = xq[4 * KP + j];
#pragma unroll
                    for (int k = 0; k < K; ++k) r = fma(xq[4 * k + j], w.th[c][k], r);
                    acc[c] = fma(r, r, acc[c]);
                }
            }
        }
    }
    // Per-chain terms that only change when sigma does: -1/(2 sigma^2) and R*(log sigma + log sqrt(2 pi)).
    struct Aux { double mhalf_inv2, rlog; };
    static constexpr int AUX_DOUBLES = 2;
    __device__ static __forceinline__ void aux_put(const Aux& a, double* p, int stride) { p[0] = a.mhalf_inv2; p[stride] = a.rlog; }
    __device__ static __forceinline__ Aux aux_get(const double* p, int stride) { Aux a; a.mhalf_inv2 = p[0]; a.rlog = p[stride]; return a; }
    template <int C, typename T>
    __device__ static __forceinline__ Aux aux(int R, const Work<C, T>& w, int c) {
        const double sg = w.sigma(c);
        Aux a;
        if (!(sg > 0.0)) {                                    // scipy: scale <= 0 -> nan
            a.mhalf_inv2 = a.rlog = __longlong_as_double(0x7ff8000000000000LL);
        } else {
            const double inv = 1.0 / sg;
            a.mhalf_inv2 = -0.5 * inv * inv;
            a.rlog = (double)R * (log(sg) + MCMCN_LOG_SQRT_2PI);
        }
        return a;
    }
    __device__ static __forceinline__ bool aux_depends_on(int p) { return p == K; }
    __device__ static __forceinline__ double finish(double acc, const Aux& a) {
        return acc * a.mhalf_inv2 - a.rlog;
    }
    template <typename T>
    __device__ static __forceinline__ double pointwise(const T* __restrict__ blk, int i, const double*, const T (&th)[P], int = 0, const void* = nullptr) {
        const T* xq = blk + (size_t)(i >> 2) * UNIT;
        const int j = i & 3;
        T r = xq[4 * KP + j];
#pragma unroll
        for (int k = 0; k < K; ++k) r = fma_t(xq[4 * k + j], th[k], r);
        const double sg = (double)th[K];
        if (!(sg > 0.0)) return __longlong_as_double(0x7ff8000000000000LL);
        const double z = (double)r / sg;
        return -0.5 * z * z - MCMCN_LOG_SQRT_2PI - log(sg);
    }
};

// Bernoulli-logit (SURVEY.md config C5): ll_i = y_i*eta_i - log(1+exp(eta_i)), eta_i = a + b*x_i.
// Block: ceil(R/4) quads of [4] x followed by [4] y.
__device__ __forceinline__ float softplus_t(float eta) {
    return fmaxf(eta, 0.0f) + __logf(1.0f + __expf(-fabsf(eta)));     // 2 MUFU per evaluation
}
__device__ __forceinline__ double softplus_t(double eta) {
    return fmax(eta, 0.0) + log1p(exp(-fabs(eta)));
}
struct Logit : NoAux {
    static constexpr int P = 2;
    static constexpr int UNIT = 8;
    static constexpr int HDR = 0;
    static constexpr int OBS_PER_UNIT = 4;
    static constexpr int FOLD_QUADS = 16;        // quads per FP64 fold of the FP32 loop

    template <typename T>
    __device__ static __forceinline__ T local(int, double v, const double*, int) { return (T)v; }
    template <int C, typename T>
    struct Work : PlainWork<P, C, T> {};

    // Whole quads, FP64 objective mode: the formula as written.
    template <int C>
    __device__ static __forceinline__ void quads(const double* __restrict__ blk, int nq, const Work<C, double>& w, double (&acc)[C]) {
        for (int q = 0; q < nq; ++q) {
            double x4[4], y4[4];
            Vec4<double>::load(blk + (size_t)q * UNIT, x4);
            Vec4<double>::load(blk + (size_t)q * UNIT + 4, y4);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const double eta = fma(w.th[c][1], x4[j], w.th[c][0]);
                    acc[c] += fma(y4[j], eta, -softplus_t(eta));
                }
            }
        }
    }
    // Whole quads, FP32 (production) mode, 16 observations per FP64 fold.  Same function, arranged for
    // the MUFU pipe that bounds it: with e = eta * log2(e) (the chain's a, b pre-scaled),
    //     y*eta - softplus(eta) = ln2 * [ (y - 1/2) e - |e|/2 - log2(1 + 2^-|e|) ]
    // and the sum of the 16 logarithms is the logarithm of the product of the 16 factors
    // (1 + 2^-|e|), each in (1, 2]: one ex2 per observation, ONE lg2 per 16 observations (was one
    // each), and four FFMA (e; product *= 1 + t; two for the linear part) instead of seven FP32 ops.
    // The product of 16 factors carries 16 roundings of 6e-8 relative, i.e. the same absolute error
    // in the logarithm as the sum of 16 rounded logarithms had.
    // Production form of the loop above: the same four FMAs and one ex2 per evaluation, issued for TWO
    // observations of one chain at a time as packed FFMA2 (e; product *= 1 + t; s += (y - 1/2) e), the pair
    // (x_j, x_j+1) being an aligned register pair of the 128-bit shared load as it is; only the |e| / 2 term
    // stays scalar (no |.| modifier on packed operands).  7 instructions per two evaluations instead of 10:
    // the loop is bound by the MUFU pipe (8 clk per warp and ex2), and the fewer issue slots the FMAs take,
    // the closer the three resident warps per scheduler keep that pipe to busy.  Even and odd observations
    // carry their own product and sum; the fold multiplies / adds the two halves before the one lg2.
    template <int C>
    __device__ static __forceinline__ void all_obs(const float* __restrict__ blk, int nobs, const Work<C, float>& w, double (&acc)[C]) {
        const int nq = nobs >> 2, rem = nobs & 3;
        f32x2 aa[C], bb[C], s2[C], pr2[C];
        const f32x2 one2 = pack2(1.0f, 1.0f), mhalf2 = pack2(-0.5f, -0.5f);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float a = w.th[c][0] * 1.4426950408889634f, b = w.th[c][1] * 1.4426950408889634f;
            aa[c] = pack2(a, a);
            bb[c] = pack2(b, b);
            s2[c] = 0ull;
            pr2[c] = one2;
        }
#define MCMCN_LOGIT_PAIR(xp, yp)                                                         \
        {                                                                                \
            const f32x2 yh = fadd2((yp), mhalf2);                                        \
            _Pragma("unroll") for (int c = 0; c < C; ++c) {                              \
                const f32x2 e2 = ffma2(bb[c], (xp), aa[c]);                              \
                float e0, e1, t0, t1, s0, s1;                                            \
                unpack2(e2, e0, e1);                                                     \
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(-fabsf(e0)));          \
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(-fabsf(e1)));          \
                pr2[c] = ffma2(pr2[c], pack2(t0, t1), pr2[c]);                           \
                unpack2(ffma2(yh, e2, s2[c]), s0, s1);                                   \
                s2[c] = pack2(fmaf(-0.5f, fabsf(e0), s0), fmaf(-0.5f, fabsf(e1), s1));   \
            }                                                                            \
        }
        // one observation: the even half only (the odd half keeps its product and sum)
#define MCMCN_LOGIT_ONE(xv, yv)                                                          \
        {                                                                                \
            const float yh = (yv) - 0.5f;                                                \
            _Pragma("unroll") for (int c = 0; c < C; ++c) {                              \
                float p0, p1, s0, s1, t;                                                 \
                unpack2(pr2[c], p0, p1);                                                 \
                unpack2(s2[c], s0, s1);                                                  \
                const float e = fmaf(lo2(bb[c]), (xv), lo2(aa[c]));                      \
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(-fabsf(e)));            \
                p0 = fmaf(p0, t, p0);                                                    \
                s0 = fmaf(-0.5f, fabsf(e), fmaf(yh, e, s0));                             \
                pr2[c] = pack2(p0, p1);                                                  \
                s2[c] = pack2(s0, s1);                                                   \
            }                                                                            \
        }
#define MCMCN_LOGIT_FOLD()                                                               \
        _Pragma("unroll") for (int c = 0; c < C; ++c) {                                  \
            float p0, p1, l;                                                             \
            unpack2(pr2[c], p0, p1);                                                     \
            asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(p0 * p1));                  \
            acc[c] += (double)(0.6931471805599453f * (sum2(s2[c]) - l));                 \
            s2[c] = 0ull;                                                                \
            pr2[c] = one2;                                                               \
        }
        // the 1-3 observations of the last, partial quad join the first fold
        const float* xr = blk + (size_t)nq * UNIT;
        if (rem & 2) MCMCN_LOGIT_PAIR(pack2(xr[0], xr[1]), pack2(xr[4], xr[5]))
        if (rem & 1) MCMCN_LOGIT_ONE(xr[rem - 1], xr[4 + rem - 1])
        // FOLD_QUADS quads per fold: one lg2 and one FP32 -> FP64 conversion (both XU operations) per
        // fold and chain.  16 quads: each half's product of up to 34 factors in (1, 2] and the product of the two
        // halves stay below 2^67; their roundings (4e-6 relative) move the logarithm by 6e-6 absolute -- against
        // group log-likelihoods of tens, inside the 1e-5 relative bar with a wide margin.
        for (int q0 = 0; q0 < nq; q0 += FOLD_QUADS) {
            const int qend = min(nq, q0 + FOLD_QUADS);
            for (int q1 = q0; q1 < qend; q1 += 4) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (q1 + u < qend) {
                        f32x2 xa, xb, ya, yb;
                        load_pairs(blk + (size_t)(q1 + u) * UNIT, xa, xb);
                        load_pairs(blk + (size_t)(q1 + u) * UNIT + 4, ya, yb);
                        MCMCN_LOGIT_PAIR(xa, ya)
                        MCMCN_LOGIT_PAIR(xb, yb)
                    }
                }
            }
            MCMCN_LOGIT_FOLD()
        }
        if (nq == 0) MCMCN_LOGIT_FOLD()
#undef MCMCN_LOGIT_PAIR
#undef MCMCN_LOGIT_ONE
#undef MCMCN_LOGIT_FOLD
    }
    template <int C>
    __device__ static __forceinline__ void all_obs(const double* __restrict__ blk, int nobs, const Work<C, double>& w, double (&acc)[C]) {
        const int nq = nobs >> 2, rem = nobs & 3;
        quads<C>(blk, nq, w, acc);
        const double* xq = blk + (size_t)nq * UNIT;
        for (int j = 0; j < rem; ++j) {
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const double eta = fma(w.th[c][1], xq[j], w.th[c][0]);
                acc[c] += fma(xq[4 + j], eta, -softplus_t(eta));
            }
        }
    }

    template <int C, typename T>
    __device__ static __forceinline__ void accumulate(const T* __restrict__ blk, int nobs, const double*,
                                                      const Work<C, T>& w, double (&acc)[C], const ObsCtx&) {
        all_obs<C>(blk, nobs, w, acc);
    }
    template <typename T>
    __device__ static __forceinline__ double pointwise(const T* __restrict__ blk, int i, const double*, const T (&th)[P], int = 0, const void* = nullptr) {
        const T* xq = blk + (size_t)(i >> 2) * UNIT;
        const T eta = fma_t(th[1], xq[i & 3], th[0]);
        return (double)fma_t(xq[4 + (i & 3)], eta, -softplus_t(eta));
    }
};

// Gaussian "distribution" objective (example/distribution.py:18-24):
//   ll_i = sum_j norm(mu_j[g(i)], sd_j).logpdf(theta_j)
// The example has no per-observation data (every row of a group is identical), but under
// complete pooling the single stepped group mixes rows of different original groups, so the
// packed record of observation i carries its own mu_j[g(i)].
// Block: ceil(R/4) quads of [4 obs][PP] mu, PP = P rounded up to 4.  obj_const = sd[P] then log(sd)[P].
template <int P_>
struct GaussDist : NoAux {
    static constexpr int P = P_;
    static constexpr int PP = (P_ + 3) & ~3;
    static constexpr int UNIT = 4 * PP;
    static constexpr int HDR = 0;
    static constexpr int OBS_PER_UNIT = 4;

    template <typename T>
    __device__ static __forceinline__ T local(int, double v, const double*, int) { return (T)v; }
    template <int C, typename T>
    struct Work : PlainWork<P, C, T> {};

    template <typename T>
    __device__ static __forceinline__ T row(const T* __restrict__ rec, const double* cst, const T (&th)[P]) {
        T v = (T)0;
#pragma unroll
        for (int j = 0; j < P; ++j) {
            const T y = (th[j] - rec[j]) / (T)cst[j];
            v = v + ((-(y * y) / (T)2 - (T)MCMCN_LOG_SQRT_2PI) - (T)cst[P + j]);
        }
        return v;
    }
    template <int C, typename T>
    __device__ static __forceinline__ void accumulate(const T* __restrict__ blk, int nobs, const double* cst,
                                                      const Work<C, T>& w, double (&acc)[C], const ObsCtx&) {
        for (int i = 0; i < nobs; ++i) {   // one evaluation per observation, summed in order (:631-633)
            const T* rec = blk + (size_t)(i >> 2) * UNIT + (i & 3) * PP;
#pragma unroll
            for (int c = 0; c < C; ++c) acc[c] = __dadd_rn(acc[c], (double)row<T>(rec, cst, w.th[c]));
        }
    }
    template <typename T>
    __device__ static __forceinline__ double pointwise(const T* __restrict__ blk, int i, const double* cst, const T (&th)[P], int = 0, const void* = nullptr) {
        return (double)row<T>(blk + (size_t)(i >> 2) * UNIT + (i & 3) * PP, cst, th);
    }
};

// User objective (north star (1), include/mcmcn.h "user objectives"): the NVRTC translation
// unit defines MCMCN_USER_P / _OBS / _HDR, `mcmc_real`, and the user's
//   __device__ mcmc_real mcmc_obj_loglik(const mcmc_real* theta, const mcmc_real* obs,
//                                        const mcmc_real* hdr, int obs_index, int group);
// before including this header.  Block: [HDR] header, then R records of OBS values.
#ifdef MCMCN_USER_P
struct UserObj : NoAux {
    static constexpr int P = MCMCN_USER_P;
    static constexpr int UNIT = MCMCN_USER_OBS;
    static constexpr int HDR = MCMCN_USER_HDR;
    static constexpr int OBS_PER_UNIT = 1;

    template <typename T>
    __device__ static __forceinline__ T local(int, double v, const double*, int) { return (T)v; }
    template <int C, typename T>
    struct Work : PlainWork<P, C, T> {};

    template <int C, typename T>
    __device__ static __forceinline__ void accumulate(const T* __restrict__ blk, int nobs, const double*,
                                                      const Work<C, T>& w, double (&acc)[C], const ObsCtx& ctx) {
        const T* hdr = reinterpret_cast<const T*>(ctx.hdr);
        for (int i = 0; i < nobs; ++i) {
#pragma unroll
            for (int c = 0; c < C; ++c)
                acc[c] += (double)mcmc_obj_loglik(w.th[c], blk + (size_t)i * UNIT, hdr, ctx.obs0 + i, ctx.group);
        }
    }
    template <typename T>
    __device__ static __forceinline__ double pointwise(const T* __restrict__ blk, int i, const double*, const T (&th)[P],
                                                       int g, const void* hdr) {
        return (double)mcmc_obj_loglik(th, blk + (size_t)i * UNIT, reinterpret_cast<const T*>(hdr), i, g);
    }
};
#endif

// ---------------------------------------------------------------- kernel arguments
struct SweepArgs {
    // model
    const void* data;
    const long long* group_off;
    const int* group_nobs;
    const int* task_group0;
    const double* obj_const;
    int P, G;
    int partial;
    int tile_cap_elems;
    int tile_bytes;               // dynamic shared memory reserved for the tile; parking slots follow
    mcmcn_prior prior[MCMCN_MAX_PARAMS];
    // state
    int n_chains, S;
    long long chain_id0;
    double* theta;
    double* scale;
    unsigned* counts;
    double* ll;
    double* lprior;
    const double* hyper;
    const double* hyper_lsd;      // hyper + 3 P S (log sd) and hyper + 4 P S (1 / sd): bases formed on the host
    const double* hyper_isd;
    // iteration
    long long iter;
    unsigned long long seed;
    int tune, count, use_override;
    StepTapes tp;
    // eval-only mode
    const double* pooled_theta;   // [P][S] or NULL
    double* out_ll;               // [G][S]
    // tensor-core path (mcmcn_tc.cuh): per-group blocks [X_hi | X_lo | NE], element offsets, stage size
    const void* tc_data;
    const long long* tc_group_off;
    int tc_stage_bytes;
    int tc_stages;                // 2: the next group's block is staged while this one is used; 1: big blocks
};

// Arguments of eval_tc_kernel (mcmcn_tc.cuh): the log-likelihood of one candidate vector per chain over a
// range of (small) groups on the tensor core -- complete pooling split over observations.
struct EvalTcArgs {
    const void* tc_data;          // operand blocks of the small groups (mcmcn_model.tc_data of the split model)
    const long long* tc_group_off;
    const int* group_nobs;
    const double* bbar;           // [K] common reference point of every small group (row 0 of the split model's obj_const)
    const double* cand;           // [P][S] candidate vector per chain
    double* part;                 // [gridDim.x][S] log-likelihood of the candidate over the CTA's group range
    int P, G, n_chains, S;
    int tc_stage_bytes;
};

// Compile-time specialisation of the step kernel.  F < 0: everything decided at run time (the
// general kernel: replay tapes, traces, groups streamed through the tile).  F >= 0: the
// production variants -- no tape, no trace, every task fits the tile -- with the pooling mode
// and the burn-in bookkeeping folded at compile time, which removes a third of the
// per-decision instructions and most of the kernel's code size.
#define MCMCN_F_PARTIAL 1
#define MCMCN_F_COUNT 2

// Stage `elems` elements starting at `src` into the tile and wait for them.
// All threads of the CTA call this; thread 0 issues the TMA bulk copy.
template <typename T>
__device__ __forceinline__ void stage_tile(T* tile, const T* src, long long elems, unsigned mb, unsigned& parity,
                                           bool need_sync) {
    if (need_sync) __syncthreads();          // previous readers of the tile are done
    if (threadIdx.x == 0) {
        const unsigned bytes = (unsigned)(elems * (long long)sizeof(T));
        mbar_expect_tx(mb, bytes);
        tma_bulk_g2s(smem_u32(tile), src, bytes, mb);
    }
    mbar_wait(mb, parity);
    parity ^= 1u;
}

// Group accumulators (Obj::finish turns them into log-likelihoods) for C chains; the group's
// block is either resident in the tile (blk != NULL) or streamed through it in chunks.
template <class Obj, int C, typename T, bool STREAM>
__device__ __forceinline__ void group_loglik(const SweepArgs& a, const T* blk, T* tile, int g, int R, unsigned mb,
                                             unsigned& parity, const typename Obj::template Work<C, T>& w,
                                             double (&acc)[C]) {
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = 0.0;
    ObsCtx ctx;
    ctx.group = g;
    ctx.obs0 = 0;
    ctx.hdr = reinterpret_cast<const T*>(a.data) + a.group_off[g];
    if (!STREAM || blk != nullptr) {
        Obj::template accumulate<C>(blk + Obj::HDR, R, a.obj_const, w, acc, ctx);
    } else {
        const T* src = reinterpret_cast<const T*>(a.data) + a.group_off[g] + Obj::HDR;
        const int unit = Obj::UNIT > 0 ? Obj::UNIT : 1;
        const int chunk_obs = (a.tile_cap_elems / unit) * Obj::OBS_PER_UNIT;
        for (int o = 0; o < R; o += chunk_obs) {
            const int n = min(chunk_obs, R - o);
            const long long elems = (long long)((n + Obj::OBS_PER_UNIT - 1) / Obj::OBS_PER_UNIT) * Obj::UNIT;
            stage_tile<T>(tile, src + (long long)(o / Obj::OBS_PER_UNIT) * Obj::UNIT, elems, mb, parity, true);
            ctx.obs0 = o;
            Obj::template accumulate<C>(tile, n, a.obj_const, w, acc, ctx);
        }
    }
}

// ---------------------------------------------------------------- the step kernel
// grid = (tasks, chain blocks); block = NW warps; one warp = 32*C chains of one group at a time.
// MINB = minimum resident CTAs per SM the register allocation must allow (2 -> at most 128 registers).
template <class Obj, int C, typename T, int MINB, int F, int MAXT = 256>
__global__ void __launch_bounds__(MAXT, MINB) sweep_kernel(const SweepArgs a) {
    constexpr int P = Obj::P;
    constexpr bool GENERAL = F < 0;
    const bool partial = GENERAL ? (a.partial != 0) : ((F & MCMCN_F_PARTIAL) != 0);
    const bool count = GENERAL ? (a.count != 0) : ((F & MCMCN_F_COUNT) != 0);
    const bool replay = GENERAL && a.tp.tape_z != nullptr;
    const bool trace = GENERAL && a.tp.tr_ll != nullptr;
    const bool forced = GENERAL && a.tp.tape_acc != nullptr;
    const bool override_lp = GENERAL && a.use_override != 0;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* tile = reinterpret_cast<T*>(smem_raw);
    __shared__ unsigned long long mbar_storage;
    const unsigned mb = smem_u32(&mbar_storage);

    const int task = blockIdx.x;
    const int g0 = a.task_group0[task], g1 = a.task_group0[task + 1];
    const long long e0 = a.group_off[g0], e1 = a.group_off[g1];
    const bool fits = !GENERAL || (e1 - e0) <= (long long)a.tile_cap_elems;
    if (threadIdx.x == 0) mbar_init(mb, 1);
    __syncthreads();
    unsigned parity = 0;
    if (fits) stage_tile<T>(tile, reinterpret_cast<const T*>(a.data) + e0, e1 - e0, mb, parity, false);

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int cbase = (blockIdx.y * nw + warp) * (32 * C) + lane;
    const size_t S = (size_t)a.S;
    // lanes past the last chain redo the last chain's work and store nothing
    int chl[C];
    bool on[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        on[c] = cbase + 32 * c < a.n_chains;
        chl[c] = min(cbase + 32 * c, a.n_chains - 1);
    }
    // per-thread parking slots in shared memory behind the tile: [field][c][thread], 8 bytes each
    double* park = reinterpret_cast<double*>(smem_raw + a.tile_bytes);
    enum { ST_PROP = 0, ST_U, ST_LPPROP, ST_LPCUR, ST_LLCUR, ST_OLD, ST_RAND2, ST_AUX };
#define SLOT(f, c) park[((f) * C + (c)) * blockDim.x + threadIdx.x]

    for (int g = g0; g < g1; ++g) {
        const int R = a.group_nobs[g];
        const T* blk = fits ? tile + (a.group_off[g] - e0) : nullptr;

        typename Obj::template Work<C, T> w;
#pragma unroll
        for (int c = 0; c < C; ++c) {
#pragma unroll
            for (int p = 0; p < P; ++p)
                w.set(c, p, Obj::template local<T>(p, a.theta[((size_t)p * a.G + g) * S + chl[c]], a.obj_const, g));
            SLOT(ST_LLCUR, c) = a.ll[(size_t)g * S + chl[c]];
            Obj::aux_put(Obj::template aux<C, T>(R, w, c), &SLOT(ST_AUX, c), C * (int)blockDim.x);
        }

#pragma unroll 1
        for (int p = 0; p < P; ++p) {
            // Decision code is written stage by stage over the C chains with selects instead of
            // branches, so the C independent dependency chains interleave in one basic block.
            // Everything that must survive the observation loop is parked in shared memory
            // (SLOT), so the loop runs spill-free and nothing after it waits on L2.
            const size_t row = ((size_t)p * a.G + g) * S;
            {
                double cur[C], sc[C], z[C], uu[C], prop[C];
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    cur[c] = a.theta[row + chl[c]];
                    sc[c] = a.scale[row + chl[c]];
                }
                if (count) {                                           // burn-in: the counters are read after the decision -- have them in L1 by then
#pragma unroll
                    for (int c = 0; c < C; ++c) prefetch_l1(a.counts + row + chl[c]);
                }
                if (p + 1 < P) {                                       // next sweep's state into L1 meanwhile
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        prefetch_l1(a.theta + row + (size_t)a.G * S + chl[c]);
                        prefetch_l1(a.scale + row + (size_t)a.G * S + chl[c]);
                        if (partial) {
                            prefetch_l1(a.hyper + ((size_t)0 * P + p + 1) * S + chl[c]);
                            prefetch_l1(a.hyper + ((size_t)3 * P + p + 1) * S + chl[c]);
                            prefetch_l1(a.hyper + ((size_t)4 * P + p + 1) * S + chl[c]);
                        }
                        else prefetch_l1(a.lprior + row + (size_t)a.G * S + chl[c]);
                    }
                }
                else if (g + 1 < g1) {                                 // last sweep of the group: the next group's state, which
#pragma unroll                                                         // the group prologue and its first sweep read, into L1
                    for (int c = 0; c < C; ++c) {
                        const size_t nx = (size_t)(g + 1) * S + chl[c];
#pragma unroll
                        for (int q = 0; q < P; ++q) prefetch_l1(a.theta + (size_t)q * a.G * S + nx);
                        prefetch_l1(a.scale + nx);
                        prefetch_l1(a.ll + nx);
                        if (count) prefetch_l1(a.counts + nx);
                        if (!partial) prefetch_l1(a.lprior + nx);
                    }
                }
                if (replay) {
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        z[c] = a.tp.tape_z[row + chl[c]];
                        uu[c] = a.tp.tape_u[row + chl[c]];
                    }
                } else if ((p & 1) == 0) {
                    // the odd sweep's draws wait in a parking slot as (float z, 32-bit word)
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const SweepDraws d = sweep_draws(a.chain_id0 + chl[c], a.seed, a.iter, p, a.G, g);
                        z[c] = (double)d.z0;
                        uu[c] = uniform_from32(d.u0);
                        SLOT(ST_RAND2, c) = __hiloint2double((int)d.u1, __float_as_int(d.z1));
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const double packed = SLOT(ST_RAND2, c);
                        z[c] = (double)__int_as_float(__double2loint(packed));
                        uu[c] = uniform_from32((unsigned)__double2hiint(packed));
                    }
                }
#pragma unroll
                for (int c = 0; c < C; ++c) prop[c] = propose(cur[c], sc[c], z[c]);
                // log-priors of the proposal and of the current value (pure functions of state
                // known now; the reference evaluates them after the likelihood, :335, :331)
                double lp_prop[C], lp_cur[C];
                if (partial) {
                    double mu[C], lsd[C], isd[C];
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        mu[c] = a.hyper[((size_t)0 * P + p) * S + chl[c]];
                        lsd[c] = a.hyper[((size_t)3 * P + p) * S + chl[c]];
                        isd[c] = a.hyper[((size_t)4 * P + p) * S + chl[c]];
                    }
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        lp_prop[c] = norm_logpdf_inv(prop[c], mu[c], isd[c], lsd[c]);
                        lp_cur[c] = override_lp ? a.lprior[row + chl[c]] : norm_logpdf_inv(cur[c], mu[c], isd[c], lsd[c]);
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        lp_prop[c] = prior_logpdf(a.prior[p], prop[c]);
                        lp_cur[c] = a.lprior[row + chl[c]];
                    }
                }
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    SLOT(ST_PROP, c) = prop[c];
                    SLOT(ST_U, c) = uu[c];
                    SLOT(ST_LPPROP, c) = lp_prop[c];
                    SLOT(ST_LPCUR, c) = lp_cur[c];
                    SLOT(ST_OLD, c) = (double)w.get(c, p);
                    w.set(c, p, Obj::template local<T>(p, prop[c], a.obj_const, g));
                }
            }

            double acc[C];
            group_loglik<Obj, C, T, GENERAL>(a, blk, tile, g, R, mb, parity, w, acc);

            typename Obj::Aux aux_prop[C];
#pragma unroll
            for (int c = 0; c < C; ++c) aux_prop[c] = Obj::aux_get(&SLOT(ST_AUX, c), C * (int)blockDim.x);
            if (Obj::aux_depends_on(p)) {
#pragma unroll
                for (int c = 0; c < C; ++c) aux_prop[c] = Obj::template aux<C, T>(R, w, c);
            }
            // decide_fast / decide_exact over C chains, written out here: the exact test is hoisted out of the
            // chain loop (one rare branch for all C chains), and its short-circuit recomputation of decide_fast's
            // `exact` keeps the observation loop's register allocation (through the function it moves by 1-4
            // registers and adds spills in some linear-regression instantiations)
            double llp[C], diff[C], uu[C], lp_prop[C], post_cur[C];
            bool acc_own[C];
            bool exact_any = false;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                uu[c] = SLOT(ST_U, c);
                lp_prop[c] = SLOT(ST_LPPROP, c);
                post_cur[c] = SLOT(ST_LPCUR, c) + SLOT(ST_LLCUR, c);
            }
#pragma unroll
            for (int c = 0; c < C; ++c) {
                llp[c] = Obj::finish(acc[c], aux_prop[c]);
                const double post_prop = lp_prop[c] + llp[c];
                diff[c] = post_prop - post_cur[c];
                const bool b1 = !finite64(post_cur[c]) && finite64(post_prop);
                const bool test = finite64(llp[c]) && finite64(diff[c]);       // branches 4/5 draw the uniform
                const int fast = log_u_vs_diff_fast(uu[c], diff[c]);
                acc_own[c] = b1 || (test && fast > 0);
                exact_any = exact_any || (!b1 && test && fast == 0);
            }
            if (exact_any) {                                           // rare: within 1e-6 of the threshold
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const bool b1 = !finite64(post_cur[c]) && finite64(lp_prop[c] + llp[c]);
                    if (!b1 && finite64(llp[c]) && finite64(diff[c]) && log_u_vs_diff_fast(uu[c], diff[c]) == 0)
                        acc_own[c] = decide_exact(uu[c], diff[c]);
                }
            }
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const size_t at = row + chl[c];
                bool accept = acc_own[c];
                if (GENERAL) accept = trace_and_force(a.tp, at, trace && on[c], forced, llp[c], lp_prop[c], diff[c], accept);
                if (accept) {                                      // :369-378, :608-610
                    if (on[c]) {
                        a.theta[at] = SLOT(ST_PROP, c);
                        if (!partial) a.lprior[at] = lp_prop[c];
                    }
                    SLOT(ST_LLCUR, c) = llp[c];
                    Obj::aux_put(aux_prop[c], &SLOT(ST_AUX, c), C * (int)blockDim.x);
                } else {
                    w.set(c, p, (T)SLOT(ST_OLD, c));
                }
                if (count && on[c]) a.counts[at] = count_and_tune(a.counts[at], accept, a.tune, a.scale + at);
            }
        }
#pragma unroll
        for (int c = 0; c < C; ++c)
            if (on[c]) a.ll[(size_t)g * S + chl[c]] = SLOT(ST_LLCUR, c);
    }
#undef SLOT
}

// Group log-likelihood of the current (or pooled) parameter values, no proposal.
template <class Obj, int C, typename T>
__global__ void __launch_bounds__(256) eval_kernel(const SweepArgs a) {
    constexpr int P = Obj::P;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* tile = reinterpret_cast<T*>(smem_raw);
    __shared__ unsigned long long mbar_storage;
    const unsigned mb = smem_u32(&mbar_storage);
    const int task = blockIdx.x;
    const int g0 = a.task_group0[task], g1 = a.task_group0[task + 1];
    const long long e0 = a.group_off[g0], e1 = a.group_off[g1];
    const bool fits = (e1 - e0) <= (long long)a.tile_cap_elems;
    if (threadIdx.x == 0) mbar_init(mb, 1);
    __syncthreads();
    unsigned parity = 0;
    if (fits) stage_tile<T>(tile, reinterpret_cast<const T*>(a.data) + e0, e1 - e0, mb, parity, false);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int cbase = (blockIdx.y * nw + warp) * (32 * C) + lane;
    const size_t S = (size_t)a.S;
    for (int g = g0; g < g1; ++g) {
        const int R = a.group_nobs[g];
        const T* blk = fits ? tile + (a.group_off[g] - e0) : nullptr;
        typename Obj::template Work<C, T> w;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int ch = min(cbase + 32 * c, a.n_chains - 1);
#pragma unroll
            for (int p = 0; p < P; ++p) {
                const double v = a.pooled_theta ? a.pooled_theta[(size_t)p * S + ch] : a.theta[((size_t)p * a.G + g) * S + ch];
                w.set(c, p, Obj::template local<T>(p, v, a.obj_const, g));
            }
        }
        double out[C];
        group_loglik<Obj, C, T, true>(a, blk, tile, g, R, mb, parity, w, out);
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int ch = cbase + 32 * c;
            if (ch < a.n_chains) a.out_ll[(size_t)g * S + ch] = Obj::finish(out[c], Obj::template aux<C, T>(R, w, c));
        }
    }
}

// Pointwise log-likelihood of the current state (saveLogLikelihood, :656-659, :907-909).
// Not a hot path: reads the blocks straight from global memory.  grid = (G, chain blocks of 128).
// The index of the group's first observation is the sum of the group sizes before it, which
// each block adds up itself (`obs_off` may be NULL), so the call needs no scratch memory.
template <class Obj, typename T>
__global__ void pointwise_kernel(const SweepArgs a, const long long* obs_off, double* out) {
    constexpr int P = Obj::P;
    __shared__ long long part[128];
    const int g = blockIdx.x;
    long long o0;
    if (obs_off) {
        o0 = obs_off[g];
    } else {
        long long s = 0;
        for (int h = threadIdx.x; h < g; h += blockDim.x) s += a.group_nobs[h];
        part[threadIdx.x] = s;
        __syncthreads();
        for (int w = 64; w > 0; w >>= 1) {
            if ((int)threadIdx.x < w && threadIdx.x + w < blockDim.x) part[threadIdx.x] += part[threadIdx.x + w];
            __syncthreads();
        }
        o0 = part[0];
    }
    const int ch = blockIdx.y * blockDim.x + threadIdx.x;
    if (ch >= a.n_chains) return;
    const size_t S = (size_t)a.S;
    T th[P];
#pragma unroll
    for (int p = 0; p < P; ++p) th[p] = Obj::template local<T>(p, a.theta[((size_t)p * a.G + g) * S + ch], a.obj_const, g);
    const T* blk = reinterpret_cast<const T*>(a.data) + a.group_off[g];
    const int R = a.group_nobs[g];
    for (int i = 0; i < R; ++i)
        out[(size_t)(o0 + i) * S + ch] = Obj::template pointwise<T>(blk + Obj::HDR, i, a.obj_const, th, g, blk);
}

// ---------------------------------------------------------------- Gibbs hyper update
// HyperParameter.update (posteriorSampling.py:463-498) + the new prior's sd / log sd
// (getDistribution :500-502).  One block = 32 chains x NS group slices for one name.
struct HyperArgs {
    int P, G, n_chains, S;
    long long chain_id0;
    const double* theta;
    double* hyper;
    long long iter;
    unsigned long long seed;
    const double* tape_zmu;     // [P][S] or NULL
    const double* tape_qsig;    // [P][S] or NULL
};

// Gamma(a, 1) by Marsaglia-Tsang on the chain's Philox stream.
__device__ inline double gamma_draw(double a, long long chain_id, unsigned long long seed, long long iter, unsigned p) {
    const bool boost = a < 1.0;
    const double aa = boost ? a + 1.0 : a;
    const double d = aa - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    double g = d;
    for (unsigned k = 0; k < 64u; ++k) {
        const uint4 r = philox_draw(chain_id, seed, iter, MCMCN_STREAM_GAMMA, p, k);
        const double x = normal_from(r.x, r.y);
        double v = 1.0 + c * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        const double u = uniform_from(r.z, r.w);
        if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) { g = d * v; break; }
    }
    if (boost) {
        const uint4 r = philox_draw(chain_id, seed, iter, MCMCN_STREAM_GAMMA, p, 1000u);
        g *= pow(uniform_from(r.x, r.y) + 1.1102230246251565e-16, 1.0 / a);
    }
    return g;
}

// The two draws of HyperParameter.update for (name p, chain ch), from the tapes when replaying: the standard
// normal of the mu draw (:487) and the unit inverse-gamma of the sigma2 draw (:497-498).
__device__ __forceinline__ double hyper_z(const HyperArgs& a, int p, int ch) {
    if (a.tape_zmu) return a.tape_zmu[(size_t)p * a.S + ch];
    const uint4 r = philox_draw(a.chain_id0 + ch, a.seed, a.iter, MCMCN_STREAM_HYPER, (unsigned)p, 0u);
    return normal_from(r.x, r.y);
}
__device__ __forceinline__ double hyper_q(const HyperArgs& a, int p, int ch) {
    if (a.tape_qsig) return a.tape_qsig[(size_t)p * a.S + ch];
    return 1.0 / gamma_draw(((double)a.G - 1.0) / 2.0, a.chain_id0 + ch, a.seed, a.iter, (unsigned)p);
}
// mu = muHat + sqrt(sigma2_old / G) z, :485-487
__device__ __forceinline__ double hyper_mu(const HyperArgs& a, int p, int ch, double muHat, double z) {
    const double sigma2_old = a.hyper[((size_t)1 * a.P + p) * a.S + ch];
    const double sd = sqrt(sigma2_old / (double)a.G);                       // :486
    return __dadd_rn(muHat, __dmul_rn(sd, z));
}
// sigma2 from the sum of squares about the new mu and the unit inverse-gamma draw q (:494-498), then the five
// rows of hyper: mu, sigma2, sd, log sd, 1 / sd (getDistribution :500-502)
__device__ __forceinline__ void hyper_finish(const HyperArgs& a, int p, int ch, double mu, double ss, double q) {
    const double n = (double)a.G;
    const double hat = ss / (n - 1.0);
    const double aa = (n - 1.0) / 2.0;
    const double sigma2 = __dadd_rn(__dmul_rn(q, __dmul_rn(aa, hat)), 0.0);
    const double sd = sqrt(sigma2);
    const size_t S = (size_t)a.S;
    a.hyper[((size_t)0 * a.P + p) * S + ch] = mu;
    a.hyper[((size_t)1 * a.P + p) * S + ch] = sigma2;
    a.hyper[((size_t)2 * a.P + p) * S + ch] = sd;
    a.hyper[((size_t)3 * a.P + p) * S + ch] = log(sd);
    a.hyper[((size_t)4 * a.P + p) * S + ch] = 1.0 / sd;
}

template <int NS>
__global__ void __launch_bounds__(32 * NS) hyper_kernel(const HyperArgs a) {
    __shared__ double red[NS][33];
    __shared__ double mu_s[32];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int ch = blockIdx.x * 32 + tx;
    const int p = blockIdx.y;
    const bool on = ch < a.n_chains;
    const size_t S = (size_t)a.S;
    const double* th = a.theta + ((size_t)p * a.G) * S + ch;
    const double n = (double)a.G;

    // pass 1: mean (numpy.mean, :485)
    double s = 0.0;
    if (on) for (int g = ty; g < a.G; g += NS) s += th[(size_t)g * S];
    red[ty][tx] = s;
    __syncthreads();
    if (ty == 0) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < NS; ++k) t += red[k][tx];
        mu_s[tx] = on ? hyper_mu(a, p, ch, t / n, hyper_z(a, p, ch)) : 0.0;
    }
    __syncthreads();
    // pass 2: sum of squares about the NEW mu (:494)
    const double mu = mu_s[tx];
    s = 0.0;
    if (on) for (int g = ty; g < a.G; g += NS) { const double d = th[(size_t)g * S] - mu; s = fma(d, d, s); }
    __syncthreads();
    red[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && on) {
        double ss = 0.0;
#pragma unroll
        for (int k = 0; k < NS; ++k) ss += red[k][tx];
        hyper_finish(a, p, ch, mu, ss, hyper_q(a, p, ch));
    }
}

// The same update with ONE read of theta, for many groups (G >= 512), where the previous
// iteration's mu is a shift c within a few standard errors of the mean: sums of (theta - c) and
// (theta - c)^2, then  mean = c + S1 / G  and
//   sum (theta - mu)^2 = (S2 - S1^2 / G) + G (mu - mean)^2     (two non-negative terms).
// Agrees with the two-pass kernel to 1e-13 relative at C3's shape (tests/test_gpu_dropin.py).
// The sums are ALWAYS taken over MCMCN_HYPER_SLICES = 16 group slices (slice j = groups j, j + 16, ... in
// order; then the 16 slices in order), whatever the launch shape, so that the result does not depend on how
// many chains a GPU holds.  Shapes: CX chains per block row (a warp row reads CX * 8 contiguous bytes of one
// group's values: 32 chains = 256 bytes per DRAM page touched measured 21.8 us at C3, 64 chains 19.1 us;
// 16,384 chains: 284 / 238 / 205 us for 32 / 64 / 128) and SPR slices per thread row (16 / SPR rows).
#define MCMCN_HYPER_SLICES 16
template <int CX, int SPR>
__global__ void __launch_bounds__(CX * (MCMCN_HYPER_SLICES / SPR)) hyper_onepass_kernel(const HyperArgs a) {
    constexpr int NS = MCMCN_HYPER_SLICES;
    __shared__ double red1[NS][CX + 1], red2[NS][CX + 1];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int ch = blockIdx.x * CX + tx;
    const int p = blockIdx.y;
    const bool on = ch < a.n_chains;
    const size_t S = (size_t)a.S;
    const double* th = a.theta + ((size_t)p * a.G) * S + ch;
    const double n = (double)a.G;
    double c = 0.0;
    if (on) {
        c = a.hyper[((size_t)0 * a.P + p) * S + ch];
        if (!finite64(c)) c = th[0];
    }
    // The two random draws of this (name, chain) do not depend on the sums: the finishing row forms them before
    // its loads, under the other rows' memory latency, instead of after the block's barrier (a serial tail of
    // Philox, Box-Muller, Marsaglia-Tsang and FP64 logarithms with the rest of the GPU idle).
    double z = 0.0, q = 0.0;
    if (ty == 0 && on) {
        z = hyper_z(a, p, ch);
        q = hyper_q(a, p, ch);
    }
#pragma unroll
    for (int q = 0; q < SPR; ++q) {
        const int slice = ty * SPR + q;
        double s1 = 0.0, s2 = 0.0;
        if (on) {
            // eight loads in flight per thread and slice (a thread reads only G / 16 values per slice: without
            // the unroll the loop is one L2 / DRAM latency per value); the sums keep their order
            const double* tq = th + (size_t)slice * S;
            const size_t step = (size_t)NS * S;
            int g = slice;
            for (; g + 7 * NS < a.G; g += 8 * NS, tq += 8 * step) {
                double v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) v[k] = tq[(size_t)k * step];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const double d = v[k] - c;
                    s1 += d;
                    s2 = fma(d, d, s2);
                }
            }
            for (; g < a.G; g += NS, tq += step) {
                const double d = *tq - c;
                s1 += d;
                s2 = fma(d, d, s2);
            }
        }
        red1[slice][tx] = s1;
        red2[slice][tx] = s2;
    }
    __syncthreads();
    if (ty == 0 && on) {
        double t1 = 0.0, t2 = 0.0;
#pragma unroll
        for (int k = 0; k < NS; ++k) { t1 += red1[k][tx]; t2 += red2[k][tx]; }
        const double dmean = t1 / n;
        const double muHat = c + dmean;                                           // numpy.mean, :485
        const double mu = hyper_mu(a, p, ch, muHat, z);
        const double dmu = mu - muHat;
        hyper_finish(a, p, ch, mu, fma(n * dmu, dmu, fmax(fma(-dmean, t1, t2), 0.0)), q);   // :494
    }
}

// ---------------------------------------------------------------- complete pooling, split over observations
// One group of all N observations (CompletePooling, posteriorSampling.py:662-685) leaves only the
// chains to parallelise over in the step kernel.  When the host provides the same observations as
// many small groups (mcmcn_model.split), a sweep of name p is three launches: propose (per chain),
// eval_kernel over the small groups with the candidate vector as pooled parameters (observations x
// chains across the GPU), decide (per chain: partial sums added in group order, then the same
// decision tree, tuning and random-number recipe as the step kernels).
struct CompleteArgs {
    int P, p, n_chains, S, n_parts;
    long long chain_id0, iter;
    unsigned long long seed;
    int tune, count;
    mcmcn_prior prior;            // of name p
    mcmcn_prior prior_next;       // of name p + 1 (decide kernel with propose_next)
    int propose_next;             // complete_decide_kernel also forms the proposal and candidate of name p + 1
    double* theta;                // [P][1][S]
    double* scale;
    unsigned* counts;
    double* ll;                   // [1][S]
    double* lprior;               // [P][1][S]
    double* cand;                 // [P][S] candidate vector: current values, name p replaced by the proposal
    double* part;                 // [n_parts][S] log-likelihood of the candidate per small group
    double* park;                 // [3][S] proposal, uniform, proposal log-prior
    StepTapes tp;                 // [P][1][S] arrays of this iteration
};

// Proposal of name p for chain c (lanes past the last chain redo its work): candidate vector, parked proposal,
// uniform and proposal log-prior.
__device__ __forceinline__ void complete_propose(const CompleteArgs& a, int p, const mcmcn_prior& prior, int c) {
    const int chl = min(c, a.n_chains - 1);
    const size_t S = (size_t)a.S, at = (size_t)p * S + chl;
    double z, u;
    if (a.tp.tape_z) {
        z = a.tp.tape_z[at];
        u = a.tp.tape_u[at];
    } else {                      // the step kernels' draws with G = 1
        const SweepDraws d = sweep_draws(a.chain_id0 + chl, a.seed, a.iter, p, 1, 0);
        z = (double)((p & 1) ? d.z1 : d.z0);
        u = uniform_from32((p & 1) ? d.u1 : d.u0);
    }
    const double prop = propose(a.theta[at], a.scale[at], z);
    for (int k = 0; k < a.P; ++k) a.cand[(size_t)k * S + c] = (k == p) ? prop : a.theta[(size_t)k * S + chl];
    a.park[c] = prop;
    a.park[S + c] = u;
    a.park[2 * S + c] = prior_logpdf(prior, prop);
}

static __global__ void __launch_bounds__(128) complete_propose_kernel(const CompleteArgs a) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.S) return;
    complete_propose(a, a.p, a.prior, c);
}

// block = (32 chains, 32 slices of the small groups): slice sums in group order, then the 32 slice
// sums in slice order -- a fixed summation order, whatever the launch
static __global__ void __launch_bounds__(1024) complete_decide_kernel(const CompleteArgs a) {
    __shared__ double slice_sum[32][33];
    const int c = blockIdx.x * 32 + threadIdx.x;                        // < S (a multiple of 32)
    const size_t S = (size_t)a.S;
    {
        const int per = (a.n_parts + 31) / 32;
        const int g0 = min((int)threadIdx.y * per, a.n_parts), g1 = min(g0 + per, a.n_parts);
        double sum = 0.0;
#pragma unroll 8
        for (int g = g0; g < g1; ++g) sum += a.part[(size_t)g * S + c];
        slice_sum[threadIdx.y][threadIdx.x] = sum;
    }
    __syncthreads();
    if (threadIdx.y != 0) return;
    if (c >= a.n_chains) {                                              // padding lanes only keep the next candidate filled
        if (a.propose_next) complete_propose(a, a.p + 1, a.prior_next, c);
        return;
    }
    const size_t at = (size_t)a.p * S + c;
    double llp = 0.0;
#pragma unroll
    for (int j = 0; j < 32; ++j) llp += slice_sum[j][threadIdx.x];
    const double prop = a.park[c], u = a.park[S + c], lp_prop = a.park[2 * S + c];
    const double post_prop = lp_prop + llp;
    const double post_cur = a.lprior[at] + a.ll[c];
    const double diff = post_prop - post_cur;
    bool exact;
    bool accept = decide_fast(post_cur, post_prop, llp, diff, u, exact);
    if (exact) accept = decide_exact(u, diff);
    accept = trace_and_force(a.tp, at, a.tp.tr_ll != nullptr, a.tp.tape_acc != nullptr, llp, lp_prop, diff, accept);
    if (accept) {                                                       // :369-378
        a.theta[at] = prop;
        a.lprior[at] = lp_prop;
        a.ll[c] = llp;
    }
    if (a.count) a.counts[at] = count_and_tune(a.counts[at], accept, a.tune, a.scale + at);
    // the next sweep's proposal in the same launch (this chain's own state only; tapes are indexed by name)
    if (a.propose_next) complete_propose(a, a.p + 1, a.prior_next, c);
}

// ---------------------------------------------------------------- retained-sample write-back
// One row of StepMethod.values (:648-654, :780-787): per name [mu, sigma2 (partial)], theta[0..G-1].
// store[(row*ncol + col)*S + chain]; a warp writes 32 consecutive chains.  grid = (columns / MCMCN_SNAP_COLS, chain blocks).
#define MCMCN_SNAP_COLS 8      /* columns per thread: eight independent loads in flight (one per thread measured 44 us per
                                  config 3 row, 2.5 TB/s) */
template <typename TS>
__global__ void snapshot_kernel(int P, int G, int partial, int n_chains, int S, const double* theta,
                                const double* hyper, TS* store_row) {
    const int ch = blockIdx.y * blockDim.x + threadIdx.x;
    const int per = G + (partial ? 2 : 0), ncol = P * per;
    const int col0 = blockIdx.x * MCMCN_SNAP_COLS;
    if (ch >= n_chains) return;
    double v[MCMCN_SNAP_COLS];
#pragma unroll
    for (int k = 0; k < MCMCN_SNAP_COLS; ++k) {
        const int col = col0 + k;
        if (col < ncol) {
            const int p = col / per, j = col - p * per;
            v[k] = (partial && j < 2) ? hyper[((size_t)j * P + p) * S + ch]
                                      : theta[((size_t)p * G + (j - (partial ? 2 : 0))) * S + ch];
        }
    }
#pragma unroll
    for (int k = 0; k < MCMCN_SNAP_COLS; ++k)
        if (col0 + k < ncol) store_row[(size_t)(col0 + k) * S + ch] = (TS)v[k];
}

// out[c] = sum_g ll[g][c] (NEGATE: its negation), from 0.0 in group order: the pooled negative log-likelihood
// (mcmcn_pooled_nll) and the complete-pooling log-likelihood over the small groups (mcmcn_group_loglik)
template <bool NEGATE>
static __global__ void group_sum_kernel(int G, int S, const double* ll, double* out) {
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= S) return;
    double s = 0.0;
    for (int g = 0; g < G; ++g) s += ll[(size_t)g * S + ch];
    out[ch] = NEGATE ? -s : s;
}

}  // namespace mcmcn
