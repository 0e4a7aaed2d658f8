// mcmcn_kernels.cu -- ahead-of-time instantiations of the step path for sm_100a and the
// C-ABI launchers declared in include/mcmcn.h.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "mcmcn_host.h"
#include "mcmcn_registry.h"

namespace mcmcn {

thread_local std::string g_last_error;

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
}

static const int kTileCapBytes = 64 * 1024;
// tcgen05 path (mcmcn_tc.cuh): two TMA stages of one group block each + the 4 KB ones operand; the
// floor keeps the CTAs at four per SM, which is what their 128 TMEM columns allow
static const int kTcStageCapBytes = 48 * 1024;       // one stage of up to 48 KB (512 observations) or two of up to 24 KB
static const int kTcSmemFloorBytes = 48 * 1024;
static const int kTcCtaSlots = 4 * 148;

struct Stamp { cudaEvent_t e0, e1; int kind; double* out; };
static thread_local std::vector<Stamp> g_stamps;

// ---------------------------------------------------------------- kernel registry
const KernelSet* user_kernel_set(const void* handle);   // mcmcn_nvrtc.cu

// AOT kernels (host stubs) and NVRTC kernels (cudaKernel_t handles) launch the same way
static cudaError_t launch_sweep(sweep_fn fn, dim3 grid, dim3 block, size_t smem, cudaStream_t stream, SweepArgs& a) {
    void* args[] = {&a};
    return cudaLaunchKernel((const void*)fn, grid, block, args, smem, stream);
}

static const KernelSet* find_set(int objective, int P, int K, int precision) {
    typedef const KernelSet* (*getter)(int*);
    static const getter getters[] = {sets_linreg_a, sets_linreg_b, sets_linreg_c, sets_linreg_d, sets_linreg_e,
                                     sets_linreg_f, sets_linreg_g, sets_linreg_h, sets_linreg_i, sets_logit, sets_gauss, sets_gauss_b};
    for (getter get : getters) {
        int n = 0;
        const KernelSet* sets = get(&n);
        for (int i = 0; i < n; ++i) {
            const KernelSet& s = sets[i];
            if (s.objective == objective && s.P == P && s.precision == precision &&
                (objective != MCMCN_OBJ_LINEAR_REGRESSION || s.K == K))
                return &s;
        }
    }
    return nullptr;
}

// ---------------------------------------------------------------- launch geometry
struct Geometry {
    bool wide, all_fit;
    int C, nw;
    dim3 grid, block;
    size_t tile_bytes;          // dynamic shared memory of the observation tile
    size_t smem;                // tile + parking slots of the step kernel
};

static int max_task_elems(const mcmcn_model* m) {
    long long mx = 0;
    for (int t = 0; t < m->n_tasks; ++t) {
        const long long e = m->group_off_host[m->task_group0_host[t + 1]] - m->group_off_host[m->task_group0_host[t]];
        if (e > mx) mx = e;
    }
    return (int)(mx > (1LL << 30) ? (1LL << 30) : mx);
}

static Geometry geometry(const KernelSet* ks, const mcmcn_model* m, int n_chains, int max_warps = 8) {
    Geometry g;
    g.wide = n_chains >= 32 * ks->c_wide;
    g.C = g.wide ? ks->c_wide : 1;
    const int per_warp = 32 * g.C;
    int warps = (n_chains + per_warp - 1) / per_warp;
    g.nw = warps < max_warps ? warps : max_warps;
    const int gy = (warps + g.nw - 1) / g.nw;
    g.grid = dim3((unsigned)m->n_tasks, (unsigned)gy, 1);
    g.block = dim3(32u * g.nw, 1, 1);
    long long bytes = (long long)max_task_elems(m) * ks->elem_bytes;
    g.all_fit = bytes <= kTileCapBytes;
    if (bytes > kTileCapBytes) bytes = kTileCapBytes;
    if (bytes < 16) bytes = 16;
    g.tile_bytes = (size_t)((bytes + 127) & ~127LL);
    g.smem = g.tile_bytes + (size_t)ks->park_doubles * g.C * g.block.x * sizeof(double);
    return g;
}

static int fill_args(SweepArgs& a, const KernelSet* ks, const mcmcn_model* m, const mcmcn_state* s) {
    memset(&a, 0, sizeof(a));
    a.data = m->data;
    a.group_off = reinterpret_cast<const long long*>(m->group_off);
    a.group_nobs = m->group_nobs;
    a.task_group0 = m->task_group0;
    a.obj_const = m->obj_const;
    a.P = m->n_params;
    a.G = m->n_groups;
    a.partial = m->pooling == MCMCN_POOL_PARTIAL;
    a.tile_cap_elems = kTileCapBytes / ks->elem_bytes;
    memcpy(a.prior, m->prior, sizeof(a.prior));
    a.n_chains = s->n_chains;
    a.S = s->stride;
    a.chain_id0 = s->chain_id0;
    a.theta = s->theta;
    a.scale = s->scale;
    a.counts = s->counts;
    a.ll = s->ll;
    a.lprior = s->lprior;
    a.hyper = s->hyper;
    a.hyper_lsd = s->hyper ? s->hyper + (size_t)3 * m->n_params * s->stride : nullptr;
    a.hyper_isd = s->hyper ? s->hyper + (size_t)4 * m->n_params * s->stride : nullptr;
    a.tc_data = m->tc_data;
    a.tc_group_off = reinterpret_cast<const long long*>(m->tc_group_off);
    return MCMCN_OK;
}

// Tensor-core launch shape: blockIdx.y = block of 128 chains, blockIdx.x = contiguous range of
// groups.  Ranges are sized so that the grid is a whole number of 2-CTA-per-SM waves when it is
// small and at most 32 groups long when it is large.
static bool tc_eligible(const mcmcn_model* m) {
    return m->objective == MCMCN_OBJ_LINEAR_REGRESSION && m->precision == 32 && m->n_coef <= 16 && m->tc_data &&
           m->tc_group_off && m->tc_max_block_floats > 0 && m->tc_max_block_floats * 4 <= kTcStageCapBytes &&
           !getenv("MCMCN_NO_TC");
}
// Does every group pad to 208 observations in the tensor-core blocks (193-208 observations)?  Read off
// the host copy of the FP32-pipe block table: a linear-regression block is ceil(R / 4) quads of
// 4 * KP + 4 elements.
static bool tc_uniform208(const mcmcn_model* m) {
    if (m->n_coef > 8) return false;                                  // one K block only (mcmcn_tc.cuh)
    const long long unit = 4LL * ((m->n_coef + 3) & ~3) + 4;
    for (int g = 0; g < m->n_groups; ++g) {
        const long long quads = (m->group_off_host[g + 1] - m->group_off_host[g]) / unit;
        if (quads < 49 || quads > 52) return false;
    }
    return true;
}
static Geometry tc_geometry(const mcmcn_model* m, int n_chains, int* stage_bytes, int* stages) {
    Geometry g;
    const int ncb = (n_chains + 127) / 128;
    const long long tasks = (long long)ncb * m->n_groups;
    int nr = m->n_groups;
    if (tasks > kTcCtaSlots) {
        const long long waves = (tasks + (long long)kTcCtaSlots * 32 - 1) / ((long long)kTcCtaSlots * 32);
        long long r = (waves * kTcCtaSlots + ncb / 2) / ncb;
        if (r < 1) r = 1;
        if (r > m->n_groups) r = m->n_groups;
        nr = (int)r;
    }
    g.wide = true; g.all_fit = true; g.C = 1; g.nw = 4;
    g.grid = dim3((unsigned)nr, (unsigned)ncb, 1);
    g.block = dim3(128, 1, 1);
    *stage_bytes = (int)((m->tc_max_block_floats * 4 + 1023) & ~1023LL);
    *stages = *stage_bytes <= 24 * 1024 ? 2 : 1;
    size_t smem = (size_t)*stages * (size_t)*stage_bytes + 4096 + 1024;
    if (smem < (size_t)kTcSmemFloorBytes) smem = kTcSmemFloorBytes;
    g.tile_bytes = g.smem = smem;
    return g;
}

static int validate(const mcmcn_model* m, const mcmcn_state* s, const KernelSet** ks) {
    if (!m || !s) { set_error("null model/state"); return MCMCN_ERR_INVALID; }
    if (m->n_params < 1 || m->n_params > MCMCN_MAX_PARAMS) { set_error("n_params %d out of range", m->n_params); return MCMCN_ERR_INVALID; }
    if (m->n_groups < 1 || m->n_tasks < 1) { set_error("empty model"); return MCMCN_ERR_INVALID; }
    if (s->n_chains < 1 || s->stride < s->n_chains || (s->stride & 31)) { set_error("bad chain count/stride %d/%d", s->n_chains, s->stride); return MCMCN_ERR_INVALID; }
    if (!m->task_group0_host || !m->group_off_host) { set_error("host task tables missing"); return MCMCN_ERR_INVALID; }
    if (m->objective == MCMCN_OBJ_USER) {
        *ks = user_kernel_set(m->user_objective);
        if (*ks && ((*ks)->P != m->n_params || (*ks)->precision != m->precision)) {
            set_error("user objective was compiled for P=%d precision=%d, model has P=%d precision=%d", (*ks)->P,
                      (*ks)->precision, m->n_params, m->precision);
            return MCMCN_ERR_INVALID;
        }
    } else {
        *ks = find_set(m->objective, m->n_params, m->n_coef, m->precision);
    }
    if (!*ks) {
        set_error("objective %d with P=%d K=%d precision=%d is not compiled in", m->objective, m->n_params, m->n_coef, m->precision);
        return MCMCN_ERR_UNSUPPORTED;
    }
    return MCMCN_OK;
}

static int set_smem_attr(const void* fn, size_t smem) {
    if (smem > 40 * 1024) CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return MCMCN_OK;
}

// Pointwise log-likelihood of the current state into out[N][S] (StepMethod.logLikelihood, :656-659).
static int launch_pointwise(const KernelSet* ks, const mcmcn_model* m, const mcmcn_state* s, double* out, cudaStream_t stream) {
    SweepArgs a;
    fill_args(a, ks, m, s);
    // the kernel derives each group's first observation index itself: no scratch, no synchronisation
    const dim3 grid((unsigned)m->n_groups, (unsigned)((s->n_chains + 127) / 128), 1);
    const long long* obs_off = nullptr;
    void* args[] = {&a, &obs_off, &out};
    CK(cudaLaunchKernel((const void*)ks->pointwise, grid, dim3(128, 1, 1), args, 0, stream));
    return MCMCN_OK;
}

// ---------------------------------------------------------------- per-iteration schedule of a run
// Burn-in bookkeeping of iteration i: tune on every tune_interval-th iteration below burn (but not 0); count
// accept / reject only up to the last such tune, since tune() is the counters' only reader.
struct IterFlags { int tune, count; };
static IterFlags iter_flags(const mcmcn_run_args* r, long long i) {
    long long last_tune = 0;
    if (r->burn > 0) last_tune = ((long long)(r->burn - 1) / r->tune_interval) * r->tune_interval;
    IterFlags f;
    f.tune = (i != 0 && i < r->burn && (i % r->tune_interval) == 0) ? 1 : 0;
    f.count = (i <= last_tune) ? 1 : 0;
    return f;
}

// The tape and trace arrays of iteration `it` of the call ([P][G][S] each, per_iter = P G S elements).
static StepTapes iter_tapes(const mcmcn_run_args* r, int it, size_t per_iter) {
    StepTapes t;
    t.tape_z = r->tape_z ? r->tape_z + it * per_iter : nullptr;
    t.tape_u = r->tape_u ? r->tape_u + it * per_iter : nullptr;
    t.tape_acc = r->tape_accept ? r->tape_accept + it * per_iter : nullptr;
    t.tr_ll = r->trace_ll ? r->trace_ll + it * per_iter : nullptr;
    t.tr_lp = r->trace_lp ? r->trace_lp + it * per_iter : nullptr;
    t.tr_diff = r->trace_diff ? r->trace_diff + it * per_iter : nullptr;
    t.tr_acc = r->trace_accept ? r->trace_accept + it * per_iter : nullptr;
    return t;
}

// Optional per-kernel timing (mcmcn_run_args.timing): every launch of kind k (0 step, 1 Gibbs, 2 snapshot) is
// counted in timing[3 + k]; on sampled iterations it is also bracketed by an event pair that
// mcmcn_timing_collect() reads later, so the call stays asynchronous.
struct KernelTimer {
    double* timing;
    cudaStream_t stream;
    bool sampled;
    void tic(int kind) {
        if (!timing) return;
        timing[3 + kind] += 1.0;
        if (!sampled) return;
        Stamp st; st.kind = kind; st.out = timing;
        cudaEventCreate(&st.e0); cudaEventCreate(&st.e1);
        cudaEventRecord(st.e0, stream);
        g_stamps.push_back(st);
    }
    void toc() { if (timing && sampled) cudaEventRecord(g_stamps.back().e1, stream); }
};

// The retained-row write of iteration i, when Sampler._loop keeps it (i >= burn and i % thin == 0, :887,
// Sampler._printLogLikelihood :890-891, :907-909): the chain state of model m (per name [mu, sigma2 (partial)],
// theta[0..G-1]) into store row `row`, and with loglik_store the pointwise log-likelihood of the same row.
static int write_retained_row(const KernelSet* ks, const mcmcn_model* m, const mcmcn_state* s, const mcmcn_run_args* r,
                              long long i, int64_t& row, KernelTimer& tm, cudaStream_t stream) {
    if (!r->store || i < r->burn || (i % r->thin) != 0) return MCMCN_OK;
    if (row >= r->store_rows) { set_error("sample store overflow at row %lld", (long long)row); return MCMCN_ERR_INVALID; }
    const bool partial = m->pooling == MCMCN_POOL_PARTIAL;
    const int ncol = m->n_params * (m->n_groups + (partial ? 2 : 0));
    const size_t S = (size_t)s->stride;
    const dim3 sg((unsigned)((ncol + MCMCN_SNAP_COLS - 1) / MCMCN_SNAP_COLS), (unsigned)((s->n_chains + 127) / 128), 1);
    tm.tic(2);
    if (r->store_dtype == 64)
        snapshot_kernel<double><<<sg, 128, 0, stream>>>(m->n_params, m->n_groups, partial ? 1 : 0, s->n_chains, s->stride,
                                                        s->theta, s->hyper, (double*)r->store + (size_t)row * ncol * S);
    else
        snapshot_kernel<float><<<sg, 128, 0, stream>>>(m->n_params, m->n_groups, partial ? 1 : 0, s->n_chains, s->stride,
                                                       s->theta, s->hyper, (float*)r->store + (size_t)row * ncol * S);
    tm.toc();
    if (r->loglik_store) {
        const int rc = launch_pointwise(ks, m, s, r->loglik_store + (size_t)row * (size_t)m->n_obs * S, stream);
        if (rc) return rc;
    }
    ++row;
    return MCMCN_OK;
}

// The split model of complete pooling at scale (mcmcn_model.split), its kernel set and the regions of
// m->split_scratch: candidate vector [P][S] | log-likelihood per small group [split->n_groups][S] | proposal,
// uniform and proposal log-prior [3][S].  e is null when m has no split model or MCMCN_NO_SPLIT is set: the
// single group of all N observations is then evaluated and stepped as it is.
struct Split {
    const mcmcn_model* e;
    const KernelSet* ks;
    double *cand, *part, *park;
};
static int resolve_split(const mcmcn_model* m, const mcmcn_state* s, Split& sp) {
    memset(&sp, 0, sizeof(sp));
    if (m->pooling != MCMCN_POOL_COMPLETE || !m->split || getenv("MCMCN_NO_SPLIT")) return MCMCN_OK;
    const mcmcn_model* e = m->split;
    const int rc = validate(e, s, &sp.ks);
    if (rc) return rc;
    if (e->n_params != m->n_params || e->n_obs != m->n_obs || e->objective != m->objective || e->precision != m->precision) {
        set_error("split model does not describe the same objective / observations");
        return MCMCN_ERR_INVALID;
    }
    if (!m->split_scratch) { set_error("split_scratch missing"); return MCMCN_ERR_INVALID; }
    sp.e = e;
    sp.cand = m->split_scratch;
    sp.part = sp.cand + (size_t)m->n_params * s->stride;
    sp.park = sp.part + (size_t)e->n_groups * s->stride;
    return MCMCN_OK;
}

// Complete pooling with the observations split into small groups (sp): per sweep propose -> eval over the
// small groups -> decide.  `mks` is the kernel set of the model m itself (pointwise log-likelihood of the
// retained rows).
static int run_complete_split(const KernelSet* mks, const mcmcn_model* m, const Split& sp, const mcmcn_state* s,
                              const mcmcn_run_args* r, cudaStream_t stream) {
    const mcmcn_model* e = sp.e;
    const KernelSet* ks = sp.ks;
    const int P = m->n_params, S = s->stride;
    SweepArgs ea;
    fill_args(ea, ks, e, s);
    ea.pooled_theta = sp.cand;
    ea.out_ll = sp.part;
    const Geometry g = geometry(ks, e, s->n_chains);
    ea.tile_bytes = (int)g.tile_bytes;
    const sweep_fn efn = g.wide ? ks->eval_wide : ks->eval_one;
    int rc = set_smem_attr((const void*)efn, g.tile_bytes);
    if (rc) return rc;
    // linear regression with FP32 observation math: the evaluation runs on the tensor core (eval_tc_kernel),
    // one partial log-likelihood per group RANGE instead of one per small group
    const bool etc = tc_eligible(e);
    EvalTcArgs ta;
    memset(&ta, 0, sizeof(ta));
    Geometry tg = g;
    eval_tc_fn tfn = nullptr;
    if (etc) {
        int sb = 0, st = 0;
        tg = tc_geometry(e, s->n_chains, &sb, &st);
        if (st < 2) tg.smem = tg.tile_bytes = (size_t)2 * sb + 4096 + 1024;     // the kernel double-buffers whatever the block size
        ta.tc_data = e->tc_data;
        ta.tc_group_off = reinterpret_cast<const long long*>(e->tc_group_off);
        ta.group_nobs = e->group_nobs;
        ta.bbar = e->obj_const;
        ta.cand = sp.cand;
        ta.part = sp.part;
        ta.P = P; ta.G = e->n_groups; ta.n_chains = s->n_chains; ta.S = S;
        ta.tc_stage_bytes = sb;
        tfn = tc_eval_kernel(e->n_coef > 8 ? 2 : 1);
        rc = set_smem_attr((const void*)tfn, tg.smem);
        if (rc) return rc;
    }

    CompleteArgs c;
    memset(&c, 0, sizeof(c));
    c.P = P; c.n_chains = s->n_chains; c.S = S; c.n_parts = etc ? (int)tg.grid.x : e->n_groups;
    c.chain_id0 = s->chain_id0; c.seed = r->seed;
    c.theta = s->theta; c.scale = s->scale; c.counts = s->counts; c.ll = s->ll; c.lprior = s->lprior;
    c.cand = sp.cand; c.part = sp.part; c.park = sp.park;
    const size_t per_iter = (size_t)P * S;                              // the one group of complete pooling
    int64_t row = r->store_row0;
    KernelTimer tm = {r->timing, stream, false};                        // launch counts only
    const unsigned nb = (unsigned)((S + 127) / 128);
    for (int it = 0; it < r->n_iter; ++it) {
        const long long i = r->iter0 + it;
        const IterFlags f = iter_flags(r, i);
        c.iter = i;
        c.tune = f.tune;
        c.count = f.count;
        c.tp = iter_tapes(r, it, per_iter);
        for (int p = 0; p < P; ++p) {                                   // StepMethod.step, :594-597
            c.p = p;
            c.prior = m->prior[p];
            if (p == 0) complete_propose_kernel<<<nb, 128, 0, stream>>>(c);       // later names: proposed by the decide launch before
            tm.tic(0);
            if (etc) {
                void* args[] = {&ta};
                CK(cudaLaunchKernel((const void*)tfn, tg.grid, tg.block, args, tg.smem, stream));
            } else {
                CK(launch_sweep(efn, g.grid, g.block, g.tile_bytes, stream, ea));
            }
            c.propose_next = p + 1 < P ? 1 : 0;
            c.prior_next = m->prior[p + 1 < P ? p + 1 : p];
            complete_decide_kernel<<<(unsigned)(S / 32), dim3(32, 32, 1), 0, stream>>>(c);
            tm.toc();
        }
        rc = write_retained_row(mks, m, s, r, i, row, tm, stream);
        if (rc) return rc;
    }
    CK(cudaGetLastError());
    return MCMCN_OK;
}

}  // namespace mcmcn

using namespace mcmcn;

extern "C" {

int mcmcn_version(void) { return MCMCN_VERSION; }
const char* mcmcn_last_error(void) { return g_last_error.c_str(); }
int mcmcn_tile_capacity_bytes(void) { return kTileCapBytes; }

int mcmcn_uses_tensor_core(const mcmcn_model* m) { return (m && tc_eligible(m)) ? 1 : 0; }

int mcmcn_supported(int objective, int n_params, int n_coef, int precision) {
    return find_set(objective, n_params, n_coef, precision) ? 1 : 0;
}

int mcmcn_run(const mcmcn_model* m, const mcmcn_state* s, const mcmcn_run_args* r, void* stream_) {
    const KernelSet* ks = nullptr;
    int rc = validate(m, s, &ks);
    if (rc) return rc;
    if (!r || r->n_iter < 0 || r->thin < 1 || r->tune_interval < 1) { set_error("bad run args"); return MCMCN_ERR_INVALID; }
    if (r->loglik_store && !r->store) { set_error("loglik_store goes with store (same rows)"); return MCMCN_ERR_INVALID; }
    if (r->tune_interval > 65535) { set_error("tune_interval %d: the accept / reject counters since the last tune are 16 bits each", r->tune_interval); return MCMCN_ERR_INVALID; }
    if ((r->tape_z == nullptr) != (r->tape_u == nullptr)) { set_error("tape_z and tape_u go together"); return MCMCN_ERR_INVALID; }
    if (r->trace_ll && !(r->trace_lp && r->trace_diff && r->trace_accept)) { set_error("trace arrays go together"); return MCMCN_ERR_INVALID; }
    const bool partial = m->pooling == MCMCN_POOL_PARTIAL;
    if (partial && !s->hyper) { set_error("partial pooling needs state.hyper"); return MCMCN_ERR_INVALID; }
    if (!partial && !s->lprior) { set_error("fixed priors need state.lprior"); return MCMCN_ERR_INVALID; }
    if (partial && m->n_groups < 2) { set_error("partial pooling needs at least 2 groups"); return MCMCN_ERR_INVALID; }
    if (partial && r->tape_z && (!r->tape_zmu || !r->tape_qsig)) { set_error("replay of partial pooling needs tape_zmu/tape_qsig"); return MCMCN_ERR_INVALID; }
    cudaStream_t stream = (cudaStream_t)stream_;
    Split sp;
    rc = resolve_split(m, s, sp);
    if (rc) return rc;
    if (sp.e) return run_complete_split(ks, m, sp, s, r, stream);

    SweepArgs a;
    fill_args(a, ks, m, s);
    // geometry: 128-thread CTAs (4 warps = 512 chains of one group), 3 per SM at 168 registers, which
    // keeps the observation loop spill-free (measured: 1.26 M chain-it/s against 1.15 M for 4 CTAs at
    // 128 registers and 1.10 M for 2 CTAs at 254)
    const bool tc = tc_eligible(m);
    int tc_stage_bytes = 0, tc_stages = 2;
    const Geometry g = tc ? tc_geometry(m, s->n_chains, &tc_stage_bytes, &tc_stages) : geometry(ks, m, s->n_chains, 4);
    a.tc_stage_bytes = tc_stage_bytes;
    a.tc_stages = tc_stages;
    // production variants (pooling mode and burn-in bookkeeping folded at compile time) when
    // there is no tape, no trace and every task fits the tile; the general kernel otherwise
    a.tile_bytes = (int)g.tile_bytes;
    const bool fast = g.wide && g.all_fit && !r->tape_z && !r->trace_ll && !r->tape_accept &&
                      !getenv("MCMCN_GENERAL");   // (the log-prior override iteration also runs general)
    if (getenv("MCMCN_DEBUG"))
        fprintf(stderr, "mcmcn_run: tc=%d fast=%d wide=%d all_fit=%d tape=%p trace=%p force=%p override=%d partial=%d smem=%zu grid=(%u,%u) block=%u\n",
                (int)tc, (int)fast, (int)g.wide, (int)g.all_fit, (const void*)r->tape_z, (void*)r->trace_ll, (const void*)r->tape_accept,
                r->use_lprior_override, (int)partial, g.smem, g.grid.x, g.grid.y, g.block.x);
    const bool u208 = tc && tc_uniform208(m);
    const int kb = m->n_coef > 8 ? 2 : 1;                             // K blocks of 8 coefficients
    const sweep_fn general = tc ? tc_sweep_kernel(-1, u208, kb) : (g.wide ? ks->sweep_wide : ks->sweep_one);
    sweep_fn fast_fn[4];
    for (int f = 0; f < 4; ++f) fast_fn[f] = tc ? tc_sweep_kernel(f, u208, kb) : ks->sweep_fast[f];
    rc = set_smem_attr((const void*)general, g.smem);
    for (int f = 0; f < 4 && !rc; ++f) rc = set_smem_attr((const void*)fast_fn[f], g.smem);
    if (rc) return rc;

    const size_t S = (size_t)s->stride;
    const size_t per_iter = (size_t)m->n_params * m->n_groups * S;
    const size_t per_iter_h = (size_t)m->n_params * S;
    int64_t row = r->store_row0;
    KernelTimer tm = {r->timing, stream, false};

    for (int it = 0; it < r->n_iter; ++it) {
        const long long i = r->iter0 + it;
        const IterFlags f = iter_flags(r, i);
        tm.sampled = (i & 7) == 0;                                     // every 8th iteration's launches are timed
        a.iter = i;
        a.seed = r->seed;
        a.tune = f.tune;
        a.count = f.count;
        a.use_override = (it == 0 && r->use_lprior_override && partial) ? 1 : 0;
        a.tp = iter_tapes(r, it, per_iter);
        const int fidx = (partial ? MCMCN_F_PARTIAL : 0) | (a.count ? MCMCN_F_COUNT : 0);
        const sweep_fn fn = (fast && !a.use_override) ? fast_fn[fidx] : general;
        tm.tic(0);
        CK(launch_sweep(fn, g.grid, g.block, g.smem, stream, a));
        tm.toc();

        if (partial) {
            HyperArgs h;
            h.P = m->n_params; h.G = m->n_groups; h.n_chains = s->n_chains; h.S = s->stride;
            h.chain_id0 = s->chain_id0; h.theta = s->theta; h.hyper = s->hyper;
            h.iter = i; h.seed = r->seed;
            h.tape_zmu = r->tape_zmu ? r->tape_zmu + it * per_iter_h : nullptr;
            h.tape_qsig = r->tape_qsig ? r->tape_qsig + it * per_iter_h : nullptr;
            const dim3 hg((unsigned)((s->n_chains + 31) / 32), (unsigned)m->n_params, 1);
            tm.tic(1);
            if (m->n_groups >= 512 && !getenv("MCMCN_HYPER_TWO_PASS"))
            {
                // the widest block row that still leaves about two blocks per SM (the sums do not depend on the shape)
                const unsigned nc = (unsigned)s->n_chains, np = (unsigned)m->n_params;
                if ((nc + 127) / 128 * np >= 296u)
                    hyper_onepass_kernel<128, 2><<<dim3((nc + 127) / 128, np, 1), dim3(128, 8, 1), 0, stream>>>(h);
                else if ((nc + 63) / 64 * np >= 144u)
                    hyper_onepass_kernel<64, 1><<<dim3((nc + 63) / 64, np, 1), dim3(64, 16, 1), 0, stream>>>(h);
                else
                    hyper_onepass_kernel<32, 1><<<dim3((nc + 31) / 32, np, 1), dim3(32, 16, 1), 0, stream>>>(h);
            }
            else if (m->n_groups >= 512) hyper_kernel<32><<<hg, dim3(32, 32, 1), 0, stream>>>(h);
            else if (m->n_groups >= 64) hyper_kernel<8><<<hg, dim3(32, 8, 1), 0, stream>>>(h);
            else hyper_kernel<1><<<hg, dim3(32, 1, 1), 0, stream>>>(h);
            tm.toc();
        }
        rc = write_retained_row(ks, m, s, r, i, row, tm, stream);
        if (rc) return rc;
    }
    CK(cudaGetLastError());
    return MCMCN_OK;
}

int mcmcn_timing_collect(void) {
    int rc = MCMCN_OK;
    for (Stamp& st : g_stamps) {
        float ms = 0.f;
        cudaError_t e = cudaEventSynchronize(st.e1);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, st.e0, st.e1);
        if (e == cudaSuccess) { st.out[st.kind] += ms; st.out[6 + st.kind] += 1.0; }
        else { set_error("timing: %s", cudaGetErrorString(e)); rc = MCMCN_ERR_CUDA; }
        cudaEventDestroy(st.e0);
        cudaEventDestroy(st.e1);
    }
    g_stamps.clear();
    return rc;
}

int mcmcn_group_loglik(const mcmcn_model* m, const mcmcn_state* s, const double* pooled_theta, double* out_ll, void* stream_) {
    const KernelSet* ks = nullptr;
    int rc = validate(m, s, &ks);
    if (rc) return rc;
    if (!out_ll) { set_error("null output"); return MCMCN_ERR_INVALID; }
    Split sp;
    rc = resolve_split(m, s, sp);
    if (rc) return rc;
    const mcmcn_model* em = m;                                          // the model whose groups are evaluated
    double* eout = out_ll;
    if (sp.e) {                 // complete pooling at scale: the small groups into split_scratch, added up below
        em = sp.e;
        ks = sp.ks;
        eout = sp.part;
        if (!pooled_theta) pooled_theta = s->theta;                     // G = 1: [P][1][S] is [P][S]
    }
    cudaStream_t stream = (cudaStream_t)stream_;
    SweepArgs a;
    fill_args(a, ks, em, s);
    a.pooled_theta = pooled_theta;
    a.out_ll = eout;
    const Geometry g = geometry(ks, em, s->n_chains);
    a.tile_bytes = (int)g.tile_bytes;
    const sweep_fn fn = g.wide ? ks->eval_wide : ks->eval_one;
    rc = set_smem_attr((const void*)fn, g.tile_bytes);
    if (rc) return rc;
    CK(launch_sweep(fn, g.grid, g.block, g.tile_bytes, stream, a));
    if (sp.e) group_sum_kernel<false><<<(s->stride + 127) / 128, 128, 0, stream>>>(sp.e->n_groups, s->stride, sp.part, out_ll);
    CK(cudaGetLastError());
    return MCMCN_OK;
}

int mcmcn_pooled_nll(int n_groups, int stride, const double* ll, double* out, void* stream_) {
    if (n_groups < 1 || stride < 1 || !ll || !out) { set_error("bad pooled_nll args"); return MCMCN_ERR_INVALID; }
    group_sum_kernel<true><<<(stride + 127) / 128, 128, 0, (cudaStream_t)stream_>>>(n_groups, stride, ll, out);
    CK(cudaGetLastError());
    return MCMCN_OK;
}

int mcmcn_pointwise_loglik(const mcmcn_model* m, const mcmcn_state* s, double* out, void* stream_) {
    const KernelSet* ks = nullptr;
    int rc = validate(m, s, &ks);
    if (rc) return rc;
    if (!out) { set_error("null output"); return MCMCN_ERR_INVALID; }
    return launch_pointwise(ks, m, s, out, (cudaStream_t)stream_);
}

}  // extern "C"

namespace mcmcn {
__global__ void philox_kat_kernel(const unsigned* c, const unsigned* k, unsigned* out) {
    const uint4 r = philox4x32_10(make_uint4(c[0], c[1], c[2], c[3]), make_uint2(k[0], k[1]));
    out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}
}  // namespace mcmcn

namespace mcmcn {
// The step path's own samplers, one draw (or pair) per thread: what the free-running kernels consume.
__global__ void debug_draws_kernel(int kind, long long n, unsigned long long seed, double a, double* out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // chain id = i, iteration 7, name/group index 3 (sweep 0 of group 3, G = 1): any fixed counter will do, the key carries i
    const SweepDraws d = sweep_draws(i, seed, 7, 0, 1, 3);
    switch (kind) {
        case MCMCN_DRAW_SWEEP_NORMALS:            // both Box-Muller branches of the sweep draw: out[2i], out[2i+1]
            out[2 * i] = (double)d.z0;
            out[2 * i + 1] = (double)d.z1;
            break;
        case MCMCN_DRAW_SWEEP_UNIFORMS:           // the two accept uniforms of the sweep draw
            out[2 * i] = uniform_from32(d.u0);
            out[2 * i + 1] = uniform_from32(d.u1);
            break;
        case MCMCN_DRAW_HYPER_NORMAL: {           // the mu draw of the Gibbs update
            const uint4 h = philox_draw(i, seed, 7, MCMCN_STREAM_HYPER, 3u, 0u);
            out[i] = normal_from(h.x, h.y);
            break;
        }
        case MCMCN_DRAW_UNIT_INVGAMMA:            // the sigma2 draw of the Gibbs update, unit scale
            out[i] = 1.0 / gamma_draw(a, i, seed, 7, 3u);
            break;
        case MCMCN_DRAW_UNIFORM53: {
            const uint4 r = philox_draw(i, seed, 7, MCMCN_STREAM_SWEEP, 3u, 1u);
            out[i] = uniform_from(r.x, r.y);
            break;
        }
        default:
            out[i] = __longlong_as_double(0x7ff8000000000000LL);
    }
}
}  // namespace mcmcn

extern "C" int mcmcn_debug_draws(int kind, int64_t n, uint64_t seed, double a, double* out, void* stream_) {
    if (n < 1 || !out || kind < 0 || kind > MCMCN_DRAW_UNIFORM53) { set_error("bad debug_draws args"); return MCMCN_ERR_INVALID; }
    debug_draws_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(kind, n, seed, a, out);
    CK(cudaGetLastError());
    return MCMCN_OK;
}

extern "C" int mcmcn_debug_philox(const void* counter, const void* key, void* out) {
    if (!counter || !key || !out) { set_error("null pointer"); return MCMCN_ERR_INVALID; }
    philox_kat_kernel<<<1, 1>>>((const unsigned*)counter, (const unsigned*)key, (unsigned*)out);
    CK(cudaDeviceSynchronize());
    return MCMCN_OK;
}
