// mcmcn_tc.cuh -- tcgen05 step kernel for the linear-regression objective (north star (2):
// "the regression linear predictor X.B, batched over chains, is the only dense contraction").
//
// Same algorithm, update order and decision tree as sweep_kernel (mcmcn_device.cuh; reference
// posteriorSampling.py:594-613, :334-383); only the evaluation of the group log-likelihood
// moves.  For one group and 128 chains the residuals of all observations are one small GEMM
//
//     D[chain][obs] = sum_k A[chain][k] * Xt[k][obs]        M = 128 chains, N = obs, K = 8
//
// issued as tcgen05.mma kind::tf32 with the accumulator in tensor memory.  FP32 accuracy comes
// from the 3xTF32 split (a = a_hi + a_lo, x = x_hi + x_lo, each part exactly representable in
// TF32): D = A_hi.X_hi + A_lo.X_hi + A_hi.X_lo, plus a fourth MMA that adds the centred
// response ne = x.bbar - y as 1 * (ne_hi + ne_mid + ne_lo), so the accumulator holds the
// residual itself (measured against FP64: 5e-7 of the largest residual, tools/tc_probe.cu).
//
//   * lanes = chains: thread t of the CTA owns TMEM lane t.  It writes its chain's
//     coefficients (A operand, tcgen05.st) and reads back its chain's row of residuals
//     (tcgen05.ld), squares and sums them with packed FFMA2 -- no cross-thread reduction.
//   * B operand: the group's observation block [X_hi | X_lo | NE], K-major, no swizzle, staged
//     in shared memory by one TMA bulk copy, double-buffered over groups.
//   * accumulator: 112 columns (observations) at a time; the chain state and random numbers of
//     the NEXT sweep are fetched while the MMAs of this sweep run.  Only column p of the A
//     operand changes per sweep (two one-column tcgen05.st).
//   * 128 TMEM columns per CTA (accumulator 112 + A_hi 8 + A_lo 8; the constant ones operand
//     of the ne MMA lives in shared memory) -> four CTAs per SM: the decision code is a chain of
//     dependent FP64 / Philox instructions, and it is the other CTAs' warps that hide it.
#pragma once

#include "mcmcn_device.cuh"

// -DMCMCN_DEBUG_BOUNDS: device-side asserts on every tensor-memory column, shared-memory stage and TMA
// extent the kernel computes (compute-sanitizer is not available on the GPU pool; build with
// `python __graft_entry__.py --debug-bounds` -> libmcmcn_debug.so, run the tests with MCMCN_LIB pointing at it).
#ifdef MCMCN_DEBUG_BOUNDS
#include <cassert>
#define MCMCN_CHECK(cond) assert(cond)
#else
#define MCMCN_CHECK(cond) ((void)0)
#endif

namespace mcmcn {

// ---------------------------------------------------------------- tcgen05 / TMEM PTX
__device__ __forceinline__ void tmem_alloc(unsigned* slot, unsigned ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free(unsigned addr, unsigned ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// 16 consecutive columns of this thread's lane
__device__ __forceinline__ void tmem_ld16(unsigned addr, unsigned (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(addr));
}
// tcgen05.wait::ld that also carries the loaded registers, so no use of them can be scheduled above it
__device__ __forceinline__ void tmem_wait_ld(unsigned (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                   "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
                 :: "memory");
}
__device__ __forceinline__ void tmem_st8(unsigned addr, const unsigned (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(addr), "r"(v[0]),
                 "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void mma_commit(unsigned mb) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mb) : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem descriptor], kind::tf32, one CTA
__device__ __forceinline__ void mma_tf32_ts(unsigned d, unsigned a, unsigned long long bdesc, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n}\n" ::"r"(d), "r"(a),
        "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// Shared-memory matrix descriptor, K-major, no swizzle: 8-row x 16-byte core matrices; the two
// 16-byte halves of K = 8 TF32 values are `lbo` bytes apart, consecutive 8-row groups `sbo` bytes.
__device__ __forceinline__ unsigned long long tc_smem_desc(unsigned addr, unsigned lbo, unsigned sbo) {
    return (unsigned long long)((addr >> 4) & 0x3FFF) | ((unsigned long long)((lbo >> 4) & 0x3FFF) << 16) |
           ((unsigned long long)((sbo >> 4) & 0x3FFF) << 32) | (1ull << 46);
}
// Instruction descriptor: D = F32, A = B = TF32, both K-major, dense
__device__ __forceinline__ unsigned tc_idesc(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(N >> 3) << 17) | ((unsigned)(M >> 4) << 24);
}
// nearest TF32 (10 explicit mantissa bits) of an FP32 value, as bits
__device__ __forceinline__ unsigned tf32_rn(float v) { return (__float_as_uint(v) + 0x1000u) & 0xFFFFE000u; }

// TMEM column map of one CTA: 128 columns -> four CTAs per SM.  KB = number of K blocks of 8 coefficients
// (1: K <= 8, 2: K = 9..16): the accumulator takes what the A operand (hi and lo parts, 8 columns per K block
// each) leaves -- 112 observations per chunk for KB = 1, 96 for KB = 2.
#define MCMCN_TC_D 0
#define MCMCN_TC_COLS 128
template <int KB> struct TcMap {
    static constexpr int CH = MCMCN_TC_COLS - 16 * KB;     /* observations (columns) of the accumulator */
    static constexpr int A_HI = CH;
    static constexpr int A_LO = CH + 8 * KB;
};
#define MCMCN_TC_THREADS 128
#define MCMCN_TC_ONES_BYTES 4096   /* [128][8] constant A operand of the ne MMA, in shared memory */

__device__ __forceinline__ void tmem_st1(unsigned addr, unsigned v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void tmem_st2(unsigned addr, unsigned v0, unsigned v1) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(v0), "r"(v1) : "memory");
}
// D[tmem] (+)= A[smem descriptor] . B[smem descriptor], kind::tf32, one CTA
__device__ __forceinline__ void mma_tf32_ss(unsigned d, unsigned long long adesc, unsigned long long bdesc, unsigned idesc,
                                            unsigned accumulate) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(d), "l"(adesc),
        "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// The 3 KB + 1 MMAs of observation chunk c of the block staged at `stage` (shared-memory address): per K
// block A_hi.X_hi + A_lo.X_hi + A_hi.X_lo, then 1.(ne_hi, ne_mid, ne_lo).  The block holds the slabs
// [X_hi block 0 .. KB-1 | X_lo block 0 .. KB-1 | NE], np * 32 bytes each.  Completion is signalled on `mbar`.
template <int KB>
__device__ __forceinline__ void tc_issue_chunk(unsigned tbase, unsigned stage, unsigned ones, int np, int c, unsigned mbar) {
    typedef TcMap<KB> M;
    const int row0 = c * M::CH;
    const int nc = min(M::CH, np - row0);
    MCMCN_CHECK(c >= 0 && row0 < np && nc >= 16 && (nc & 15) == 0 && nc <= M::CH);               // accumulator columns
    MCMCN_CHECK(MCMCN_TC_D + nc <= M::A_HI && M::A_LO + 8 * KB <= MCMCN_TC_COLS);
    MCMCN_CHECK((stage & 1023u) == 0u && (ones & 1023u) == 0u);                                    // descriptor bases
    const unsigned idesc = tc_idesc(128, nc);
    const unsigned slab = (unsigned)np * 32u;
    const unsigned base = stage + (unsigned)row0 * 32u;
    const unsigned d = tbase + MCMCN_TC_D;
#pragma unroll
    for (int kb = 0; kb < KB; ++kb) {
        const unsigned long long xhi = tc_smem_desc(base + kb * slab, 128, 256), xlo = tc_smem_desc(base + (KB + kb) * slab, 128, 256);
        mma_tf32_ts(d, tbase + M::A_HI + 8 * kb, xhi, idesc, kb ? 1 : 0);                         // A_hi . X_hi
        mma_tf32_ts(d, tbase + M::A_LO + 8 * kb, xhi, idesc, 1);                                  // A_lo . X_hi
        mma_tf32_ts(d, tbase + M::A_HI + 8 * kb, xlo, idesc, 1);                                  // A_hi . X_lo
    }
    mma_tf32_ss(d, tc_smem_desc(ones, 128, 256), tc_smem_desc(base + 2 * KB * slab, 128, 256), idesc, 1);   // 1 . (ne_hi, ne_mid, ne_lo)
    mma_commit(mbar);
}

#define MCMCN_TC_CONSUME(v, s)                                                    \
    _Pragma("unroll") for (int k = 0; k < 8; ++k) {                               \
        f32x2 r;                                                                  \
        asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(v[2 * k]), "r"(v[2 * k + 1])); \
        s[k & 3] = ffma2(r, r, s[k & 3]);                                         \
    }

// Sum of squares of PIECES x 16 accumulator columns of this thread's lane, fully unrolled: the
// load of piece j + 1 is in flight while piece j is squared (FFMA2, four FP32 pair accumulators).
template <int PIECES>
__device__ __forceinline__ double tc_sum_squares_fixed(unsigned addr) {
    f32x2 s[4] = {0ull, 0ull, 0ull, 0ull};
    unsigned v[2][16];
    tmem_ld16(addr, v[0]);
    tmem_wait_ld(v[0]);
#pragma unroll
    for (int j = 0; j < PIECES; ++j) {
        if (j + 1 < PIECES) tmem_ld16(addr + 16 * (j + 1), v[(j + 1) & 1]);
        MCMCN_TC_CONSUME(v[j & 1], s)
        if (j + 1 < PIECES) tmem_wait_ld(v[(j + 1) & 1]);
    }
    return (double)((sum2(s[0]) + sum2(s[1])) + (sum2(s[2]) + sum2(s[3])));
}
// The same with the four FP32 pair accumulators kept by the caller (they carry over both chunks of a
// 208-observation group: 26 terms each before the one fold into FP64).
template <int PIECES>
__device__ __forceinline__ void tc_accumulate_fixed(unsigned addr, f32x2 (&s)[4]) {
    unsigned v[2][16];
    tmem_ld16(addr, v[0]);
    tmem_wait_ld(v[0]);
#pragma unroll
    for (int j = 0; j < PIECES; ++j) {
        if (j + 1 < PIECES) tmem_ld16(addr + 16 * (j + 1), v[(j + 1) & 1]);
        MCMCN_TC_CONSUME(v[j & 1], s)
        if (j + 1 < PIECES) tmem_wait_ld(v[(j + 1) & 1]);
    }
}
__device__ __forceinline__ void tc_accumulate_any(unsigned addr, int pieces, f32x2 (&s)[4]) {
    unsigned va[16];
    for (int j = 0; j < pieces; ++j) {
        tmem_ld16(addr + 16 * j, va);
        tmem_wait_ld(va);
        MCMCN_TC_CONSUME(va, s)
    }
}
__device__ __forceinline__ double tc_sum_squares_any(unsigned addr, int pieces) {
    f32x2 s[4] = {0ull, 0ull, 0ull, 0ull};
    unsigned va[16];
    for (int j = 0; j < pieces; ++j) {
        tmem_ld16(addr + 16 * j, va);
        tmem_wait_ld(va);
        MCMCN_TC_CONSUME(va, s)
    }
    return (double)((sum2(s[0]) + sum2(s[1])) + (sum2(s[2]) + sum2(s[3])));
}
__device__ __forceinline__ double tc_sum_squares(unsigned addr, int pieces) {
    switch (pieces) {
        case 7: return tc_sum_squares_fixed<7>(addr);
        case 6: return tc_sum_squares_fixed<6>(addr);
        default: return tc_sum_squares_any(addr, pieces);
    }
}

// What a sweep reads from the chain state and the random stream; none of it depends on the
// decisions of earlier sweeps of the same iteration, so it is fetched one sweep ahead.
struct TcInputs {
    double cur, sc, z, u;
    double bbar;                    // reference point of this coefficient (0 for sigma)
    double h_mu, h_lsd, h_isd;      // partial pooling: this name's hyper-parameters
    double lp_cur;                  // fixed priors / log-prior override: stored log-prior of the current value
    unsigned cnt;                   // burn-in: accepted | rejected << 16 since the last tune, fetched with the rest (not after the decision)
};

// The odd sweep's (z, u) of sweep_draws, carried over from the even sweep.
struct TcStash { double z, u; };

// `at` = element index of (name p, group g, this chain) in the [P][G][S] arrays, `hy` = p * S + chain
// in the [5][P][S] hyper-parameters, `bb` = g * K + p in bbar; the caller bumps them per sweep.
// State loads and random numbers are separate so that they can sit behind different MMAs.
template <bool GENERAL>
__device__ __forceinline__ void tc_fetch_state(TcInputs& o, const SweepArgs& a, int p, size_t at, size_t hy, size_t bb,
                                               bool partial, bool override_lp, bool count = false) {
    const int P = a.P;
    o.cnt = count ? a.counts[at] : 0u;
    o.cur = a.theta[at];
    o.sc = a.scale[at];
    o.h_mu = o.h_lsd = o.h_isd = o.lp_cur = 0.0;
    o.bbar = p < P - 1 ? a.obj_const[bb] : 0.0;
    if (partial) {
        o.h_mu = a.hyper[hy];
        o.h_lsd = a.hyper_lsd[hy];
        o.h_isd = a.hyper_isd[hy];
        if (GENERAL && override_lp) o.lp_cur = a.lprior[at];
    } else {
        o.lp_cur = a.lprior[at];
    }
}
template <bool GENERAL>
__device__ __forceinline__ void tc_fetch_random(TcInputs& o, const SweepArgs& a, int p, int g, int chl, size_t at, bool replay,
                                                TcStash& stash) {
    if (GENERAL && replay) {
        o.z = a.tp.tape_z[at];
        o.u = a.tp.tape_u[at];
    } else if ((p & 1) == 0) {
        const SweepDraws d = sweep_draws(a.chain_id0 + chl, a.seed, a.iter, p, a.G, g);
        o.z = (double)d.z0;
        stash.z = (double)d.z1;
        o.u = uniform_from32(d.u0);
        stash.u = uniform_from32(d.u1);
    } else {
        o.z = stash.z;
        o.u = stash.u;
    }
}

// LinReg::Aux of a sigma: m = -1/(2 sigma^2), r = R (log sigma + log sqrt(2 pi)); sigma <= 0 -> nan (scipy).
// FP32 reciprocal and logarithm (1 ulp each: 1e-7 relative on the log-likelihood) in place of about
// 60 FP64 instructions for the division and the logarithm: 0.2855 -> 0.2781 ms per C3 launch.
__device__ __forceinline__ void tc_sigma_terms(double sigma, int R, double& m, double& r) {
    const float sf = (float)sigma;
    if (!(sf > 0.0f)) {
        m = r = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    const double inv = (double)__frcp_rn(sf);
    m = -0.5 * inv * inv;
    r = (double)R * ((double)logf(sf) + MCMCN_LOG_SQRT_2PI);
}

// CTA-wide rendezvous before an MMA issue: every lane's tensor-memory traffic (tcgen05.st of the
// A operand, tcgen05.ld of the accumulator) is ordered before the barrier, thread 0 issues after
// it.  (A rendezvous on a shared-memory atomic where the last warp to arrive issues and nobody
// waits measured 7 % slower: atom.acq_rel costs a MEMBAR per warp.)
__device__ __forceinline__ bool tc_rendezvous_issuer() {
    tc_fence_before();
    __syncthreads();
    bool issuer = false;
    if (threadIdx.x < 32) {                   // warp-uniform branch, then one elected lane: lets ptxas keep the
        unsigned pred;                        // MMA operands in uniform registers without a per-instruction loop
        asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
        issuer = pred != 0;
        if (issuer) tc_fence_after();
    }
    return issuer;
}

// CTA prologue of the tcgen05 kernels, called by every thread: three mbarriers ([0..1] TMA stage full, [2]
// accumulator full), the constant A operand of the ne MMA, and the CTA's MCMCN_TC_COLS tensor-memory columns.
struct TcCta {
    unsigned ones, stage0;        // shared-memory addresses of the ones operand and of TMA stage 0 (1024-byte aligned)
    unsigned tbase, tlane;        // the CTA's first TMEM column; the same with this warp's lane field (32 * warp)
    unsigned mb_tma0, mb_mma;     // mbarrier of stage 0 (stage s: + 8 s) and of the accumulator
};
__device__ __forceinline__ TcCta tc_cta_begin(unsigned char* smem_raw, unsigned long long (&mbar_s)[3], unsigned* tmem_base_s) {
    const int tid = threadIdx.x, warp = tid >> 5;
    TcCta t;
    t.ones = (smem_u32(smem_raw) + 1023u) & ~1023u;
    t.stage0 = t.ones + MCMCN_TC_ONES_BYTES;
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 3; ++i) mbar_init(smem_u32(&mbar_s[i]), 1);
    }
    {   // constant A operand of the ne MMA: every row (1, 1, 1, 0 | 0, 0, 0, 0), K-major core matrices
        for (int i = tid; i < MCMCN_TC_ONES_BYTES / 16; i += MCMCN_TC_THREADS) {
            const float one = ((i >> 3) & 1) == 0 ? 1.0f : 0.0f;      // 8 rows x 16 bytes per K half
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(t.ones + 16u * i), "f"(one), "f"(one), "f"(one), "f"(0.0f) : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor core reads
    }
    if (warp == 0) tmem_alloc(tmem_base_s, MCMCN_TC_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    t.tbase = *tmem_base_s;
    t.tlane = t.tbase + ((unsigned)warp << 21);
    t.mb_tma0 = smem_u32(&mbar_s[0]);
    t.mb_mma = smem_u32(&mbar_s[2]);
    asm volatile("" : "+r"(t.mb_tma0), "+r"(t.mb_mma));              // held in registers (else rebuilt from SR_CgaCtaId at every wait)
    return t;
}
// CTA epilogue: every tensor-memory access of the CTA is done before warp 0 frees its columns
__device__ __forceinline__ void tc_cta_end(const TcCta& t) {
    tmem_wait_st();
    tc_fence_before();
    __syncthreads();
    if ((threadIdx.x >> 5) == 0) tmem_free(t.tbase, MCMCN_TC_COLS);
}

// grid = (group ranges, chain blocks of 128); block = 128 threads; dynamic shared memory =
// the constant ones operand + a.tc_stages (2, or 1 for big groups) stages of a.tc_stage_bytes (1024-byte aligned).
// UNIFORM208: every group of the model pads to 208 observations (193-208, BASELINE config 3's 200): the
// read-back is written for exactly two accumulator chunks of 112 + 96 columns.  Otherwise groups of
// 113-224 observations take the same straight-line path with the second chunk looped, the rest the
// chunk loop.  (One kernel with all three paths measured 2.4 % slower on the 208 case.)
// KB: K blocks of 8 coefficients (2 for K = 9..16: 7 MMAs per chunk of 96 observations; UNIFORM208 is a KB = 1 path).
template <int F, bool UNIFORM208, int KB = 1>
__global__ void __launch_bounds__(MCMCN_TC_THREADS, 4) sweep_tc_kernel(const SweepArgs a) {
    static_assert(KB == 1 || !UNIFORM208, "the straight-line 112 + 96 read-back is for one K block");
    typedef TcMap<KB> M;
    constexpr int CH = M::CH;
    constexpr bool GENERAL = F < 0;
    const bool partial = GENERAL ? (a.partial != 0) : ((F & MCMCN_F_PARTIAL) != 0);
    const bool count = GENERAL ? (a.count != 0) : ((F & MCMCN_F_COUNT) != 0);
    const bool replay = GENERAL && a.tp.tape_z != nullptr;
    const bool trace = GENERAL && a.tp.tr_ll != nullptr;
    const bool forced = GENERAL && a.tp.tape_acc != nullptr;
    const bool override_lp = GENERAL && a.use_override != 0;
    const int P = a.P, K = a.P - 1;

    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ unsigned long long mbar_s[3];          // [0..1] TMA stage full, [2] accumulator full
    __shared__ unsigned tmem_base_s;

    const int nr = gridDim.x;
    const int g0 = (int)(((long long)a.G * blockIdx.x) / nr), g1 = (int)(((long long)a.G * (blockIdx.x + 1)) / nr);
    if (g0 >= g1) return;

    const int tid = threadIdx.x;
    const TcCta t = tc_cta_begin(smem_raw, mbar_s, &tmem_base_s);
    const float* tc = reinterpret_cast<const float*>(a.tc_data);
    auto stage_group = [&](int s, int g) {                             // thread 0 only
        const long long e0 = a.tc_group_off[g], e1 = a.tc_group_off[g + 1];
        const unsigned bytes = (unsigned)((e1 - e0) * 4);
        MCMCN_CHECK(s >= 0 && s < a.tc_stages && g >= g0 && g < g1);
        MCMCN_CHECK(bytes > 0 && (bytes & 15u) == 0u && (int)bytes <= a.tc_stage_bytes && ((e0 * 4) & 15) == 0);   // TMA extent
        mbar_expect_tx(t.mb_tma0 + 8u * s, bytes);
        tma_bulk_g2s(t.stage0 + (unsigned)s * (unsigned)a.tc_stage_bytes, tc + e0, bytes, t.mb_tma0 + 8u * s);
    };
    if (tid == 0) {
        stage_group(0, g0);
        if (a.tc_stages > 1 && g0 + 1 < g1) stage_group(1, g0 + 1);
    }

    const int ch = blockIdx.y * MCMCN_TC_THREADS + tid;
    const bool on = ch < a.n_chains;
    const int chl = min(ch, a.n_chains - 1);                           // lanes past the last chain redo its work, store nothing
    const size_t S = (size_t)a.S;
    unsigned tma_phase = 0, mma_phase = 0;
    TcStash stash;
    stash.z = stash.u = 0.0;

    for (int g = g0; g < g1; ++g) {
        const int s = a.tc_stages > 1 ? ((g - g0) & 1) : 0;
        const int R = a.group_nobs[g];
        const int np = max(16, (R + 15) & ~15);                        // padded observation count of the block
        const int nchunks = (np + CH - 1) / CH;
        MCMCN_CHECK(R >= 0 && np * 32 * (2 * KB + 1) == (int)((a.tc_group_off[g + 1] - a.tc_group_off[g]) * 4));   // 2 KB + 1 slabs of [np][8] floats
        MCMCN_CHECK(np * 32 * (2 * KB + 1) <= a.tc_stage_bytes && (t.tbase & 0xFFFFu) + MCMCN_TC_COLS <= 512u);
        MCMCN_CHECK(K >= 1 && K <= 8 * KB);
        const unsigned stage = t.stage0 + (unsigned)s * (unsigned)a.tc_stage_bytes;
        const double* bbar = a.obj_const + (size_t)g * K;

        const size_t GS = (size_t)a.G * S;
        size_t at = (size_t)g * S + chl, hy = (size_t)chl, bb = (size_t)g * K;   // sweep 0; bumped by GS / S / 1 per sweep
        TcInputs in;
        tc_fetch_state<GENERAL>(in, a, 0, at, hy, bb, partial, override_lp, count);
        tc_fetch_random<GENERAL>(in, a, 0, g, chl, at, replay, stash);
        const double* tg = a.theta + at;                               // (name 0, group g, this chain); name k is k * GS further
        if (g + 1 < g1) {                                              // next group's state: DRAM -> L2 meanwhile
            const double* pf = tg + S;
            for (int k = 0; k < P; ++k, pf += GS) asm volatile("prefetch.global.L2 [%0];" ::"l"(pf));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(a.ll + at + S));
        }
        // The proposal of a sweep and its centred FP32 value are formed at the end of the sweep before
        // (here: for sweep 0), so that column p (the value kept) and column p + 1 (the next proposal) of
        // the A operand go out in one two-column store.
        double prop = propose(in.cur, in.sc, in.z);
        float wcur = (float)__dsub_rn(in.cur, in.bbar), wprop = (float)__dsub_rn(prop, in.bbar);
        {   // A operand of the current state: centred coefficients (FP32), split hi / lo, 8 columns per K block
            const double* tk = tg;
#pragma unroll
            for (int kb = 0; kb < KB; ++kb) {
                unsigned hi[8], lo[8];
#pragma unroll
                for (int j = 0; j < 8; ++j, tk += GS) {
                    const int k = 8 * kb + j;
                    float b = k < K ? (float)__dsub_rn(*tk, bbar[k]) : 0.0f;
                    if (k == 0) b = wprop;                             // column 0 already holds sweep 0's proposal
                    hi[j] = tf32_rn(b);
                    lo[j] = tf32_rn(b - __uint_as_float(hi[j]));
                }
                tmem_st8(t.tlane + M::A_HI + 8 * kb, hi);
                tmem_st8(t.tlane + M::A_LO + 8 * kb, lo);
            }
        }
        double aux_m, aux_r;                                           // LinReg::Aux of the current sigma
        tc_sigma_terms(tg[(size_t)K * GS], R, aux_m, aux_r);
        double ll_cur = a.ll[at];
        mbar_wait(t.mb_tma0 + 8u * s, (tma_phase >> s) & 1u);
        tma_phase ^= 1u << s;

#pragma unroll 1
        for (int p = 0; p < P; ++p, at += GS, hy += S, ++bb) {
            const bool is_sigma = p == K;
            // log-priors of the proposal (formed at the end of the sweep before) and of the current value
            // (pure functions of state known before the sweep; the reference evaluates them after the
            // likelihood, :335, :331).  (Moving the priors or the random numbers
            // behind the MMAs instead measured 7-10 % slower, twice.)
            double lp_prop, lp_cur;
            if (partial) {
                lp_prop = norm_logpdf_inv(prop, in.h_mu, in.h_isd, in.h_lsd);
                lp_cur = (GENERAL && override_lp) ? in.lp_cur : norm_logpdf_inv(in.cur, in.h_mu, in.h_isd, in.h_lsd);
            } else {
                lp_prop = prior_logpdf(a.prior[p], prop);
                lp_cur = in.lp_cur;
            }
            const double u = in.u;
            const unsigned cnt_now = in.cnt;
            double m_prop = aux_m, r_prop = aux_r;
            const float wcur_now = wcur, wprop_now = wprop;            // this sweep's; wcur / wprop move on to the next below
            if (is_sigma) tc_sigma_terms(prop, R, m_prop, r_prop);     // LinReg::aux of the proposed sigma
            tmem_wait_st();
            if (tc_rendezvous_issuer()) tc_issue_chunk<KB>(t.tbase, stage, t.ones, np, 0, t.mb_mma);
            // while the tensor core works: state and random numbers of the next sweep.  (Drawing the
            // random numbers inside the read-back code instead, to fill its tensor-memory latency, cost
            // registers and measured 8 % slower.)
            if (p + 1 < P) {
                tc_fetch_state<GENERAL>(in, a, p + 1, at + GS, hy + S, bb + 1, partial, override_lp, count);
                tc_fetch_random<GENERAL>(in, a, p + 1, g, chl, at + GS, replay, stash);
            }

            double acc = 0.0;
            if (UNIFORM208 && np == 208) {                             // 112 + 96 observations (C3's groups): straight line, one fold
                f32x2 sq[4] = {0ull, 0ull, 0ull, 0ull};
                mbar_wait(t.mb_mma, mma_phase);
                tc_fence_after();
                tc_accumulate_fixed<7>(t.tlane + MCMCN_TC_D, sq);
                if (tc_rendezvous_issuer()) tc_issue_chunk<KB>(t.tbase, stage, t.ones, np, 1, t.mb_mma);
                mbar_wait(t.mb_mma, mma_phase ^ 1u);
                tc_fence_after();
                tc_accumulate_fixed<6>(t.tlane + MCMCN_TC_D, sq);
                acc = (double)((sum2(sq[0]) + sum2(sq[1])) + (sum2(sq[2]) + sum2(sq[3])));
            } else if (!UNIFORM208 && KB == 1 && nchunks == 2) {       // any group of 113-224 observations: the same, second chunk looped
                f32x2 sq[4] = {0ull, 0ull, 0ull, 0ull};
                mbar_wait(t.mb_mma, mma_phase);
                tc_fence_after();
                tc_accumulate_fixed<7>(t.tlane + MCMCN_TC_D, sq);
                if (tc_rendezvous_issuer()) tc_issue_chunk<KB>(t.tbase, stage, t.ones, np, 1, t.mb_mma);
                mbar_wait(t.mb_mma, mma_phase ^ 1u);
                tc_fence_after();
                tc_accumulate_any(t.tlane + MCMCN_TC_D, (np - CH) >> 4, sq);
                acc = (double)((sum2(sq[0]) + sum2(sq[1])) + (sum2(sq[2]) + sum2(sq[3])));
            } else
            for (int c = 0; c < nchunks; ++c) {
                mbar_wait(t.mb_mma, mma_phase);
                mma_phase ^= 1u;
                tc_fence_after();
                const int nc = min(CH, np - c * CH);
                acc += tc_sum_squares(t.tlane + MCMCN_TC_D, nc >> 4);
                if (c + 1 < nchunks) {                                 // the accumulator is free once every lane has read it
                    if (tc_rendezvous_issuer()) tc_issue_chunk<KB>(t.tbase, stage, t.ones, np, c + 1, t.mb_mma);
                }
            }

            const double llp = acc * m_prop - r_prop;
            const double post_prop = lp_prop + llp;
            const double post_cur = lp_cur + ll_cur;
            const double diff = post_prop - post_cur;
            bool exact;
            bool accept = decide_fast(post_cur, post_prop, llp, diff, u, exact);
            if (exact) accept = decide_exact(u, diff);                 // rare: within 1e-6 of the threshold
            if (GENERAL) accept = trace_and_force(a.tp, at, trace && on, forced, llp, lp_prop, diff, accept);
            if (accept) {                                              // :369-378, :608-610
                if (on) {
                    a.theta[at] = prop;
                    if (!partial) a.lprior[at] = lp_prop;
                }
                ll_cur = llp;
                aux_m = m_prop;
                aux_r = r_prop;
            }
            if (!is_sigma) {                                           // column p <- the value the chain keeps, column p + 1 <- the next proposal
                const float wkeep = accept ? wprop_now : wcur_now;
                const unsigned h = tf32_rn(wkeep), l = tf32_rn(wkeep - __uint_as_float(h));
                prop = propose(in.cur, in.sc, in.z);                   // `in` holds sweep p + 1 by now
                MCMCN_CHECK(p >= 0 && p < 8 * KB && p < K);                             // A-operand column
                if (p + 1 < K) {
                    wcur = (float)__dsub_rn(in.cur, in.bbar);
                    wprop = (float)__dsub_rn(prop, in.bbar);
                    const unsigned nh = tf32_rn(wprop);
                    tmem_st2(t.tlane + M::A_HI + p, h, nh);
                    tmem_st2(t.tlane + M::A_LO + p, l, tf32_rn(wprop - __uint_as_float(nh)));
                } else {                                               // the next sweep is sigma's: no column of its own
                    tmem_st1(t.tlane + M::A_HI + p, h);
                    tmem_st1(t.tlane + M::A_LO + p, l);
                }
            }
            if (count && on) a.counts[at] = count_and_tune(cnt_now, accept, a.tune, a.scale + at);
        }
        if (on) a.ll[(size_t)g * S + chl] = ll_cur;
        // every MMA that read this stage has completed (all threads waited on its mbarrier)
        if (tid == 0 && g + a.tc_stages < g1) stage_group(s, g + a.tc_stages);
    }
    tc_cta_end(t);
}

// ---------------------------------------------------------------- complete pooling: evaluation on the tensor core
// Complete pooling split over observations (mcmcn_model.split; CompletePooling, posteriorSampling.py:662-685):
// every chain evaluates ONE candidate vector over all N observations, handed over as many small groups.
// The candidate does not depend on the group, and the small groups share one reference point (the pooled
// least-squares fit), so the A operand -- the chain's centred coefficients, split hi / lo -- is written to
// tensor memory once per CTA; then per group: TMA stage, 3 KB + 1 MMAs per chunk, read-back of the chain's
// own row of residuals, sum of squares (FP32 pairs folded into FP64 per chunk).  The sum of squares of the
// CTA's whole group range is finished once: part[range][chain] = S m - N_range (log sigma + log sqrt(2 pi)).
// grid = (group ranges, chain blocks of 128); block = 128 threads; 128 TMEM columns -> four CTAs per SM.
template <int KB>
__global__ void __launch_bounds__(MCMCN_TC_THREADS, 4) eval_tc_kernel(const EvalTcArgs a) {
    typedef TcMap<KB> M;
    constexpr int CH = M::CH;
    const int K = a.P - 1;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ unsigned long long mbar_s[3];          // [0..1] TMA stage full, [2] accumulator full
    __shared__ unsigned tmem_base_s;

    const int nr = gridDim.x;
    const int g0 = (int)(((long long)a.G * blockIdx.x) / nr), g1 = (int)(((long long)a.G * (blockIdx.x + 1)) / nr);
    const int tid = threadIdx.x;
    const TcCta t = tc_cta_begin(smem_raw, mbar_s, &tmem_base_s);
    const float* tc = reinterpret_cast<const float*>(a.tc_data);
    auto stage_group = [&](int s, int g) {                             // thread 0 only
        const long long e0 = a.tc_group_off[g], e1 = a.tc_group_off[g + 1];
        const unsigned bytes = (unsigned)((e1 - e0) * 4);
        MCMCN_CHECK(s >= 0 && s < 2 && g >= g0 && g < g1);
        MCMCN_CHECK(bytes > 0 && (bytes & 15u) == 0u && (int)bytes <= a.tc_stage_bytes && ((e0 * 4) & 15) == 0);
        mbar_expect_tx(t.mb_tma0 + 8u * s, bytes);
        tma_bulk_g2s(t.stage0 + (unsigned)s * (unsigned)a.tc_stage_bytes, tc + e0, bytes, t.mb_tma0 + 8u * s);
    };
    if (tid == 0 && g0 < g1) {
        stage_group(0, g0);
        if (g0 + 1 < g1) stage_group(1, g0 + 1);
    }

    const int ch = blockIdx.y * MCMCN_TC_THREADS + tid;
    const bool on = ch < a.n_chains;
    const int chl = min(ch, a.n_chains - 1);
    const size_t S = (size_t)a.S;
    {   // A operand: the candidate's centred coefficients (FP32), split hi / lo, 8 columns per K block
        const double* ck = a.cand + chl;
#pragma unroll
        for (int kb = 0; kb < KB; ++kb) {
            unsigned hi[8], lo[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int k = 8 * kb + j;
                const float b = k < K ? (float)__dsub_rn(ck[(size_t)k * S], a.bbar[k]) : 0.0f;
                hi[j] = tf32_rn(b);
                lo[j] = tf32_rn(b - __uint_as_float(hi[j]));
            }
            tmem_st8(t.tlane + M::A_HI + 8 * kb, hi);
            tmem_st8(t.tlane + M::A_LO + 8 * kb, lo);
        }
    }
    double aux_m, aux_r1;                                              // -1/(2 sigma^2); log sigma + log sqrt(2 pi) (per observation)
    tc_sigma_terms(a.cand[(size_t)K * S + chl], 1, aux_m, aux_r1);
    tmem_wait_st();

    unsigned tma_phase = 0, mma_phase = 0;
    double acc = 0.0;
    long long nobs = 0;
    for (int g = g0; g < g1; ++g) {
        const int s = (g - g0) & 1;
        const int R = a.group_nobs[g];
        const int np = max(16, (R + 15) & ~15);
        const int nchunks = (np + CH - 1) / CH;
        const unsigned stage = t.stage0 + (unsigned)s * (unsigned)a.tc_stage_bytes;
        MCMCN_CHECK(np * 32 * (2 * KB + 1) == (int)((a.tc_group_off[g + 1] - a.tc_group_off[g]) * 4));
        nobs += R;
        mbar_wait(t.mb_tma0 + 8u * s, (tma_phase >> s) & 1u);
        tma_phase ^= 1u << s;
        for (int c = 0; c < nchunks; ++c) {
            // every lane has read the accumulator of the chunk before (and, the first time, written its A operand)
            if (tc_rendezvous_issuer()) tc_issue_chunk<KB>(t.tbase, stage, t.ones, np, c, t.mb_mma);
            mbar_wait(t.mb_mma, mma_phase);
            mma_phase ^= 1u;
            tc_fence_after();
            const int nc = min(CH, np - c * CH);
            acc += tc_sum_squares(t.tlane + MCMCN_TC_D, nc >> 4);
        }
        // every MMA that read this stage has completed (all threads waited on its mbarrier)
        if (tid == 0 && g + 2 < g1) stage_group(s, g + 2);
    }
    if (on) a.part[(size_t)blockIdx.x * S + ch] = acc * aux_m - (double)nobs * aux_r1;
    tc_cta_end(t);
}

}  // namespace mcmcn
