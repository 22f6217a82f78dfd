/*
 * qo_cuda.cu -- contexts, plans and the compute entry points of libqo100net.
 * Everything numerical happens in the kernels of qo_lumped.cuh / qo_ustrip.cuh;
 * this file compiles networks into device programs, owns HBM buffers and
 * launches.  There is no CPU evaluation path: without a device every compute
 * call returns QO_ERR_NO_DEVICE.
 */
#include <cuda_runtime.h>
#include <time.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <chrono>
#include <vector>

#include "qo_internal.h"
#include "qo_ctx_internal.h"
#include "qo_lumped.cuh"
#include "qo_ladder.cuh"
#include "qo_ladder_launch.h"
#include "qo_tf.cuh"
#include "qo_tf_launch.h"
#include "qo_ts.cuh"
#include "qo_spot.cuh"
#include "qo_tf_fs.cuh"
#include "qo_ustrip.cuh"
#include "qo_ustrip_board.cuh"
#include "qo_cpl_core.h"
#include "qo_chain_jit.h"
#include "qo_overrides.h"

static int nccl_load(NcclApi *a)
{
    memset(a, 0, sizeof *a);
    const char *names[] = { "libnccl.so.2", "libnccl.so", NULL };
    const char *why = NULL;
    for (int i = 0; names[i] && !a->h; i++) {
        a->h = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
        if (!a->h && !why) why = dlerror();            /* read it now: the next dl* call clears it */
    }
    if (!a->h) { qo_set_error("libnccl.so.2 not loadable: %s", why ? why : "dlopen failed"); return 0; }
    a->CommInitAll = (int (*)(ncclComm_t *, int, const int *))dlsym(a->h, "ncclCommInitAll");
    a->CommDestroy = (int (*)(ncclComm_t))dlsym(a->h, "ncclCommDestroy");
    a->AllReduce = (int (*)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(a->h, "ncclAllReduce");
    a->GroupStart = (int (*)(void))dlsym(a->h, "ncclGroupStart");
    a->GroupEnd = (int (*)(void))dlsym(a->h, "ncclGroupEnd");
    a->GetErrorString = (const char *(*)(int))dlsym(a->h, "ncclGetErrorString");
    if (!(a->CommInitAll && a->CommDestroy && a->AllReduce && a->GroupStart && a->GroupEnd)) { qo_set_error("libnccl lacks a required entry point"); return 0; }
    return 1;
}
enum { QO_NCCL_UINT64 = 5, QO_NCCL_SUM = 0 };   /* ncclUint64, ncclSum (nccl.h enum values) */

#define QO_TICKET_BYTES (16 + 256 * sizeof(unsigned int))
static const size_t QO_NOTAB = ~(size_t)0;
static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

/* A plan's device tables, built once on the host in one buffer: each table is a zeroed region at a 256-byte-aligned offset,
 * and every device of the ctx gets the same bytes at the same offsets */
struct QoLayout {
    std::vector<unsigned char> buf;
    size_t add(size_t bytes) { const size_t at = align256(buf.size()); buf.resize(at + bytes, 0); return at; }
    template <typename T> T *host(size_t off) { return off == QO_NOTAB ? NULL : (T *)(buf.data() + off); }
};

/* Byte offsets of a plan's tables in its device allocation; QO_NOTAB (where every offset starts): the plan's kernel does not read
 * that table.  Two grid points per entry, in the plan's precision: w2, wi2 (1/w), wsq2 (w^2), m2 (spec bits); cpl: sin/cos of the
 * coupler's nominal even/odd mode angles, or the row vector [1 Rs] M of a measured two-port in front; sblk, sdet: measured blocks'
 * ABCD per (block, point), product of their determinants per point.  The transfer-function kernel's tables, padded to whole
 * iterations: yt = -(w/wref)^2, xt = w/wref, wt = w, fu2 = the second row vector [1 -Rs] M (|S11| specs), mb = per-point byte
 * masks, itm = per-iteration (OR, AND) of the spec bits.  The counters and the ticket area follow the uploaded tables. */
struct QoTables {
    size_t prog, w2, wi2, wsq2, m2, cpl[4], sblk, sdet, fgrid, mask, yt, xt, wt, fu2[4], mb, itm, counters, ticket;
    QoTables() { memset(this, 0xFF, sizeof *this); }
};

/* mem: the tables of qo_plan::lay, then the counters, then the ticket area; fs_mem: the tables of the FULL_S flavour of the
 * transfer-function kernel (qo_plan::fs_lay) */
struct DevPlan { unsigned char *mem, *fs_mem; };

/* the kernel a plan launches, in order of precedence (select_kernel); launch-time refinements: thread-per-sample inside launch_tf,
 * the compiled chain kernel inside launch_lumped, the FULL_S transfer-function kernel ahead of them all (plan_launch_dev) */
enum QoKern { K_BOARD, K_GENERIC, K_SPOT, K_TF, K_LADDER, K_LUMPED };
static const char *const qo_kern_name[] = { "qo_mc_board_kernel", "qo_mc_generic_kernel", "qo_mc_spot_kernel", "qo_mc_tf_kernel",
                                            "qo_mc_ladder_kernel", "qo_mc_lumped_kernel" };

struct qo_plan {
    qo_ctx *ctx;
    DevProg hp;                /* host copy of the program */
    int nf, npairs, ncnt, precision, mode, generic;
    QoOverrides ov;                                       /* the environment overrides as they were at plan creation */
    QoKern kern;
    /* launch-time decisions of the transfer-function kernels, taken once at plan creation */
    int tf_cpl_matched, tf_cpl_lin, ts_ok;
    int ts_screen_ran;                                    /* the last thread-per-sample launch was qo_mc_ts_screen_kernel */
    double tf_cpl_dw1;                                    /* angular-frequency step of one grid point on a uniformly spaced grid */
    int lad_n, lad_first, lad_cpl;                        /* straight-line ladder kernel (qo_ladder.cuh) */
    int cpl_fast, cpl_same;                               /* coupler block: small-angle table path, equal mode angles */
    int spot_el0, spot_nel;                               /* spot-frequency kernel (qo_spot.cuh): <= 8 points per sample */
    TfPlan tfp;                                           /* transfer-function kernel (qo_tf.cuh): polynomial lengths, denominator form, self-check result */
    int tf_pp, tf_niter;                                  /* pairs per thread per iteration; iterations per sample */
    int fs_state;                                         /* FULL_S transfer-function path: 0 not analysed yet, 1 selected, -1 refused */
    TfPlan fsp;
    int fs_niter;
    QoLayout fs_lay;                                      /* its tables, built at the first launch that takes it */
    size_t fs_yt, fs_xt;
    int cj_debug, cj_failed[2];                           /* run-time compiled chain kernel (qo_chain_jit.h), used as ov.chain says */
    const void *cj[2];                                    /* its QcjEntry for the reduce-only / FULL_S flavour once this process holds it */
    std::string cj_src[2];
    unsigned long long cj_hash[2];
    const char *kernel_name;
    double flops_per_eval;
    int launches;
    QoLayout lay;                                         /* the tables the plan's kernel reads (qo_mc_run re-sends them on a cache hit) */
    QoTables tab;
    unsigned char *pinned;                                /* page-locked copy of lay, made the first time the tables are re-sent */
    DevPlan d[8];
    std::vector<double> f;
    std::vector<unsigned char> maskv;
    /* device address of a table on device g; NULL when the plan's kernel does not read it */
    template <typename T> T *dev(int g, size_t off) const { return off == QO_NOTAB ? NULL : (T *)(d[g].mem + off); }
    unsigned long long *counters(int g) const { return dev<unsigned long long>(g, tab.counters); }
    unsigned long long *ticket(int g) const { return dev<unsigned long long>(g, tab.ticket); }
};

static void tf_launch_setup(qo_plan *p, const QoOverrides *ov);

/* ---- ctx ---------------------------------------------------------------- */
static int devctx_init(DevCtx *d, int device)
{
    memset(d, 0, sizeof *d);
    d->device = device;
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
    d->own_stream = 1;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    d->sm_count = prop.multiProcessorCount;
    CU(cudaEventCreate(&d->ev0));
    CU(cudaEventCreate(&d->ev1));
    /* plans and sweeps allocate their (small) device tables stream-ordered; keep up to 256 MB of freed blocks in the
     * device's pool so that a one-shot call does not pay cudaMalloc/cudaFree (~1 ms per nominal sweep before) */
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long thr = 256ull << 20;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    } else cudaGetLastError();
    return QO_OK;
}

static int device_count(int *n)
{
    cudaError_t e = cudaGetDeviceCount(n);
    if (e != cudaSuccess || *n <= 0) {
        cudaGetLastError();
        qo_set_error("no usable CUDA device (%s); libqo100net has no CPU fallback", e == cudaSuccess ? "count is 0" : cudaGetErrorString(e));
        return QO_ERR_NO_DEVICE;
    }
    return QO_OK;
}

extern "C" int qo_ctx_create_on_device(int device, qo_ctx **out)
{
    qo_clear_error();
    if (!out || device < 0) return QO_ERR_ARG;
    int n, rc = device_count(&n);
    if (rc) return rc;
    if (device >= n) { qo_set_error("device %d out of range (%d visible)", device, n); return QO_ERR_ARG; }
    qo_ctx *c = (qo_ctx *)calloc(1, sizeof(qo_ctx));
    if (!c) return QO_ERR_NOMEM;
    c->ndev = 1;
    rc = devctx_init(&c->d[0], device);
    if (rc) { qo_ctx_destroy(c); return rc; }          /* releases whatever the partial initialisation created */
    *out = c;
    return QO_OK;
}

extern "C" int qo_ctx_create(int ngpus, qo_ctx **out)
{
    qo_clear_error();
    if (!out || !(ngpus == 1 || ngpus == 2 || ngpus == 4 || ngpus == 8)) { qo_set_error("ngpus must be 1, 2, 4 or 8"); return QO_ERR_ARG; }
    int n, rc = device_count(&n);
    if (rc) return rc;
    if (ngpus > n) { qo_set_error("%d GPUs requested, %d visible", ngpus, n); return QO_ERR_NO_DEVICE; }
    qo_ctx *c = (qo_ctx *)calloc(1, sizeof(qo_ctx));
    if (!c) return QO_ERR_NOMEM;
    c->ndev = ngpus;
    for (int g = 0; g < ngpus; g++) {
        rc = devctx_init(&c->d[g], g);
        if (rc) { qo_ctx_destroy(c); return rc; }
    }
    if (ngpus > 1) {
        /* the only collective on this path: one all-reduce of the u64 counters */
        if (!nccl_load(&c->nccl)) { qo_ctx_destroy(c); return QO_ERR_NCCL; }      /* nccl_load has set the error text */
        int devs[8];
        for (int g = 0; g < ngpus; g++) devs[g] = g;
        c->have_nccl = 1;                              /* from here on qo_ctx_destroy also destroys the communicators that exist */
        int r = c->nccl.CommInitAll(c->comm, ngpus, devs);
        if (r != 0) { qo_set_error("ncclCommInitAll: %s", c->nccl.GetErrorString ? c->nccl.GetErrorString(r) : "?"); qo_ctx_destroy(c); return QO_ERR_NCCL; }
    }
    *out = c;
    return QO_OK;
}

extern "C" int qo_ctx_set_stream(qo_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return QO_ERR_ARG;
    DevCtx *d = &ctx->d[0];
    CU(cudaSetDevice(d->device));
    if (ctx->mc_cache) { cudaStreamSynchronize(d->stream); qo_plan_destroy(ctx->mc_cache); ctx->mc_cache = NULL; }
    if (d->own_stream) { cudaStreamDestroy(d->stream); d->own_stream = 0; }
    if (cuda_stream) d->stream = (cudaStream_t)cuda_stream;
    else { CU(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking)); d->own_stream = 1; }
    return QO_OK;
}

extern "C" int qo_ctx_num_devices(const qo_ctx *ctx) { return ctx ? ctx->ndev : QO_ERR_ARG; }

extern "C" void qo_ctx_destroy(qo_ctx *ctx)
{
    if (!ctx) return;
    if (ctx->mc_cache) { qo_plan_destroy(ctx->mc_cache); ctx->mc_cache = NULL; }
    for (int g = 0; g < ctx->ndev; g++) {
        cudaSetDevice(ctx->d[g].device);
        if (ctx->have_nccl && ctx->comm[g]) ctx->nccl.CommDestroy(ctx->comm[g]);
        if (ctx->d[g].own_stream && ctx->d[g].stream) cudaStreamDestroy(ctx->d[g].stream);
        if (ctx->d[g].ev0) cudaEventDestroy(ctx->d[g].ev0);
        if (ctx->d[g].ev1) cudaEventDestroy(ctx->d[g].ev1);
    }
    cudaGetLastError();                                /* a partially built ctx may hand invalid handles to the calls above */
    free(ctx);
}

/* ---- network -> device program ------------------------------------------ */
static int touches(const qo_mc_cfg *cfg, int elem, int param)
{
    if (!cfg) return 0;
    for (int i = 0; i < cfg->n_tol; i++)
        if (cfg->tol[i].elem == elem && cfg->tol[i].param == param && cfg->tol[i].tol != 0.0) return 1;
    return 0;
}

/* ALG-v1 algorithmic flops per eval (SURVEY §8d): immittance + chain step per element, +26 for ABCD->|S|^2 */
static double alg_flops(int opcode)
{
    switch (opcode) {
    case OP_SER_R: case OP_SHUNT_G: return 0 + 8;
    case OP_SER_L: case OP_SER_C: case OP_SHUNT_C: case OP_SHUNT_L: return 1 + 8;
    case OP_SER_LCS: case OP_SHUNT_LCP: return 3 + 8;
    case OP_SER_LCP: case OP_SHUNT_LCS: return 4 + 8;
    case OP_SER_LOSSY_L: case OP_SHUNT_LOSSY_L: return 17 + 16;
    case OP_SER_LOSSY_C: return 3 + 16;
    case OP_SHUNT_LOSSY_C: return 9 + 16;
    case OP_TLINE: return 56 + 10;
    case OP_CPL: return 56 + 40;
    case OP_SBLOCK: return 56;
    default: return 0;
    }
}

static int build_prog(const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec, const qo_mc_cfg *cfg,
                      DevProg *hp, int *generic, double *flops, std::vector<unsigned char> *mask)
{
    memset(hp, 0, sizeof *hp);
    if (cfg && cfg->mode != QO_MODE_REDUCE_ONLY && cfg->mode != QO_MODE_FULL_S) { qo_set_error("unknown mode %d (QO_MODE_REDUCE_ONLY | QO_MODE_FULL_S)", cfg->mode); return QO_ERR_ARG; }
    if (cfg && cfg->precision != 0 && cfg->precision != 32 && cfg->precision != 64) { qo_set_error("precision must be 64 or 32 (0 = 64), not %d", cfg->precision); return QO_ERR_ARG; }
    if (net->n > QO_MAX_OPS) { qo_set_error("network has %d elements, limit %d", net->n, QO_MAX_OPS); return QO_ERR_RANGE; }
    if (nspec < 0 || nspec > QO_NSPEC_MAX) { qo_set_error("at most %d specs", QO_NSPEC_MAX); return QO_ERR_RANGE; }
    hp->n_ops = net->n;
    hp->cplms_elem = hp->cplms_sub = -1;
    int last_sub = -1;
    hp->rs = net->rs; hp->rl = net->rl; hp->rsrl = net->rs * net->rl; hp->k21 = 2.0 * sqrt(net->rs * net->rl);
    hp->seed = cfg ? cfg->seed : 0;
    hp->dist = cfg ? cfg->dist : 0;
    if (hp->dist != QO_DIST_UNIFORM && hp->dist != QO_DIST_GAUSS3S) { qo_set_error("unknown distribution %d", hp->dist); return QO_ERR_ARG; }
    int coff = 0, ustrip = 0, trig = 0;
    double fl = 26.0;
    for (int e = 0; e < net->n; e++) {
        const qo_elem *el = &net->e[e];
        for (int k = 0; k < 6; k++) { hp->nom[e][k] = el->p[k]; hp->tvar[e][k] = -1; }
        hp->kind[e] = el->kind;
        int op = OP_NOP, nco = 0;
        int lossy = el->p[1] != 0.0 || el->p[2] != 0.0 || touches(cfg, e, 1) || touches(cfg, e, 2);
        switch (el->kind) {
        case QO_SER_R: op = OP_SER_R; nco = 1; break;
        case QO_SHUNT_R: op = OP_SHUNT_G; nco = 1; break;
        case QO_SER_L: op = lossy ? OP_SER_LOSSY_L : OP_SER_L; nco = lossy ? 4 : 1; break;
        case QO_SHUNT_L: op = lossy ? OP_SHUNT_LOSSY_L : OP_SHUNT_L; nco = lossy ? 4 : 1; break;
        case QO_SER_C: op = lossy ? OP_SER_LOSSY_C : OP_SER_C; nco = lossy ? 4 : 1; break;
        case QO_SHUNT_C: op = lossy ? OP_SHUNT_LOSSY_C : OP_SHUNT_C; nco = lossy ? 4 : 1; break;
        case QO_SER_LC_SER: op = OP_SER_LCS; nco = 2; break;
        case QO_SER_LC_PAR: op = OP_SER_LCP; nco = 2; break;
        case QO_SHUNT_LC_SER: op = OP_SHUNT_LCS; nco = 2; break;
        case QO_SHUNT_LC_PAR: op = OP_SHUNT_LCP; nco = 2; break;
        case QO_TLINE: op = OP_TLINE; nco = 3; trig = 1; break;
        case QO_CPL_THRU: op = OP_CPL; nco = 8; trig = 1; break;
        case QO_SBLOCK:
            op = OP_SBLOCK; nco = 1; trig = 1;
            if (!(el->p[0] >= 0 && el->p[0] < net->nblk)) { qo_set_error("element %d: S-parameter block %g is not in the net", e, el->p[0]); return QO_ERR_ARG; }
            break;
        case QO_SUBST: op = OP_SUBST; last_sub = e; break;        /* a substrate alone does not make the network microstrip */
        case QO_CPL_MS:
            /* physical coupled line: compiled to the coupled-line opcode; its electrical parameters come per sample
             * from the pre-pass (qo_cplms_kernel) */
            if (last_sub < 0) { qo_set_error("element %d: QO_CPL_MS needs a preceding QO_SUBST", e); return QO_ERR_ARG; }
            if (hp->cplms_elem >= 0) { qo_set_error("element %d: at most one QO_CPL_MS per network", e); return QO_ERR_UNSUPPORTED; }
            op = OP_CPL; nco = 8; trig = 1;
            hp->cplms_elem = e; hp->cplms_sub = last_sub;
            break;
        case QO_MLIN: op = OP_MLIN; ustrip = 1; break;
        case QO_MCORN: op = OP_MCORN; ustrip = 1; break;
        case QO_MTEE: op = OP_MTEE; ustrip = 1; break;
        case QO_MOPEN: op = OP_MOPEN; ustrip = 1; break;
        default: qo_set_error("element %d: unsupported kind %d", e, el->kind); return QO_ERR_UNSUPPORTED;
        }
        hp->opcode[e] = op;
        hp->coff[e] = coff;
        coff += (nco + 1) & ~1;          /* keep every record 16-byte aligned */
        fl += alg_flops(op);
    }
    if (coff > QO_MAX_COEF) { qo_set_error("coefficient table too large"); return QO_ERR_RANGE; }
    hp->n_coef = coff;
    hp->has_trig = trig;
    hp->has_ustrip = ustrip;
    if (hp->cplms_elem >= 0) {
        if (ustrip) { qo_set_error("QO_CPL_MS cannot be mixed with MLIN/MCORN/MTEE/MOPEN elements yet"); return QO_ERR_UNSUPPORTED; }
        const qo_elem *c = &net->e[hp->cplms_elem], *sb = &net->e[hp->cplms_sub];
        qo_cpl_core(c->p[0], c->p[1], sb->p[1], sb->p[2], sb->p[0], c->p[3], c->p[4], c->p[2], hp->cplms_nom);
        if (!isfinite(hp->cplms_nom[0]) || !isfinite(hp->cplms_nom[1])) { qo_set_error("QO_CPL_MS: geometry outside the analysis model's range"); return QO_ERR_RANGE; }
    }
    if (!ustrip)            /* substrates that only serve a QO_CPL_MS take no part in the chain */
        for (int e = 0; e < net->n; e++) if (hp->opcode[e] == OP_SUBST) hp->opcode[e] = OP_NOP;
    hp->op0 = 0;
    while (hp->op0 < net->n - 1 && hp->opcode[hp->op0] == OP_NOP) hp->op0++;
    *generic = ustrip;
    *flops = ustrip ? 0.0 : fl;

    /* tolerances -> per (element, parameter) random variable */
    int nvar = 0;
    if (cfg) {
        if (cfg->n_tol < 0 || (cfg->n_tol > 0 && !cfg->tol)) return QO_ERR_ARG;
        for (int i = 0; i < cfg->n_tol; i++) {
            const qo_tol *t = &cfg->tol[i];
            if (t->elem < 0 || t->elem >= net->n || t->param < 0 || t->param >= 6) { qo_set_error("tolerance %d: element/param out of range", i); return QO_ERR_ARG; }
            if (t->var < 0 || t->var >= QO_MAX_VAR) { qo_set_error("tolerance %d: random variable index must be in [0,%d)", i, QO_MAX_VAR); return QO_ERR_RANGE; }
            if (hp->tvar[t->elem][t->param] >= 0) { qo_set_error("tolerance %d: parameter perturbed twice", i); return QO_ERR_ARG; }
            hp->tvar[t->elem][t->param] = (int16_t)t->var;
            hp->tmode[t->elem][t->param] = (uint8_t)(t->mode == QO_TOL_ABS);
            hp->ttol[t->elem][t->param] = t->tol;
            if (t->var + 1 > nvar) nvar = t->var + 1;
        }
    }
    hp->n_var = nvar;

    /* specs -> canonical linear thresholds + per-frequency bit mask */
    hp->nspec = nspec;
    mask->assign((size_t)nf + 1, 0);
    for (int s = 0; s < nspec; s++) {
        const qo_spec *sp = &spec[s];
        double lin = pow(10.0, sp->limit / 10.0);
        hp->spec_user_kind[s] = sp->kind;
        hp->spec_limit[s] = sp->limit;
        switch (sp->kind) {
        case QO_SPEC_S21_MIN_DB: hp->spec_kind[s] = SK_DEN2_MAX; hp->spec_thr[s] = ustrip ? lin : hp->k21 * hp->k21 / lin; break;
        case QO_SPEC_S21_MAX_DB: hp->spec_kind[s] = SK_DEN2_MIN; hp->spec_thr[s] = ustrip ? lin : hp->k21 * hp->k21 / lin; break;
        case QO_SPEC_S11_MAX_DB: hp->spec_kind[s] = SK_S11_MAX; hp->spec_thr[s] = lin; hp->need_s11 = 1; break;
        case QO_SPEC_S22_MAX_DB: hp->spec_kind[s] = SK_S22_MAX; hp->spec_thr[s] = lin; hp->need_s22 = 1; break;
        case QO_SPEC_MU_MIN: {      /* limit dimensionless; mu from all four S-parameters, so the 2x2 product (need_s11) */
            if (ustrip) { qo_set_error("QO_SPEC_MU_MIN is not available for microstrip networks"); return QO_ERR_UNSUPPORTED; }
            if (cfg && cfg->precision == 32) { qo_set_error("QO_SPEC_MU_MIN needs FP64 (1 - |S11|^2 near |S11| = 1)"); return QO_ERR_UNSUPPORTED; }
            int blk = 0;
            for (int e = 0; e < net->n; e++) blk |= net->e[e].kind == QO_SBLOCK;
            if (!blk) { qo_set_error("QO_SPEC_MU_MIN needs a measured two-port (QO_SBLOCK): every other element is passive, mu >= 1"); return QO_ERR_ARG; }
            hp->spec_kind[s] = SK_MU_MIN; hp->spec_thr[s] = sp->limit; hp->need_s11 = 1;
            break;
        }
        case QO_SPEC_GD_MAX:        /* limit in seconds; evaluated in-kernel by the central difference of arg S21 */
            if (ustrip) { qo_set_error("QO_SPEC_GD_MAX is not available for microstrip networks"); return QO_ERR_UNSUPPORTED; }
            for (int e = 0; e < net->n; e++)
                if (net->e[e].kind == QO_SBLOCK) { qo_set_error("QO_SPEC_GD_MAX is not available for networks with measured blocks"); return QO_ERR_UNSUPPORTED; }
            hp->spec_kind[s] = SK_GD_MAX; hp->spec_thr[s] = sp->limit; hp->need_gd |= 1 << s;
            break;
        default: qo_set_error("spec %d: unknown kind %d", s, sp->kind); return QO_ERR_ARG;
        }
        int hits = 0;
        for (int k = 0; k < nf; k++)
            if (f[k] >= sp->f_lo && f[k] <= sp->f_hi) { (*mask)[k] |= (unsigned char)(1u << s); hits++; }
        if (cfg && cfg->hist_bins > 0 && cfg->hist_spec == s && hits == 0) { qo_set_error("histogram spec %d covers no grid frequency", s); return QO_ERR_ARG; }
    }
    if (cfg && cfg->hist_bins > 0) {
        if (!qo_hist_cfg_ok(cfg, nspec)) return QO_ERR_ARG;
        hp->hist_bins = cfg->hist_bins; hp->hist_spec = cfg->hist_spec; hp->hist_lo = cfg->hist_lo; hp->hist_hi = cfg->hist_hi;
    }
    return QO_OK;
}

/* The straight-line ladder kernel covers: reduce-only FP64 jobs whose specs are on |S21| and |S11|, on a
 * network that is an alternating series-inductor / shunt-capacitor ladder of 1..11 elements
 * (pcb/generic-filter), optionally behind one coupled-line block.  QO100NET_KERNEL=interp forces the
 * opcode interpreter (A/B runs, parity tests of both paths). */
static int ladder_eligible(const DevProg *hp, int mode, int precision, const QoOverrides *ov, int *n, int *first, int *cpl)
{
    if (ov->kernel == QoOverrides::INTERP) return 0;
    if (mode != QO_MODE_REDUCE_ONLY || hp->need_gd) return 0;
    if (precision == 32 && hp->need_s11) return 0;          /* FP32 mode: |S21| specs only on the straight-line kernel */
    if (hp->nspec > QO_LAD_NSPEC || hp->n_var > QO_MAX_VAR) return 0;
    for (int s = 0; s < hp->nspec; s++)
        if (hp->spec_kind[s] != SK_DEN2_MAX && hp->spec_kind[s] != SK_DEN2_MIN && hp->spec_kind[s] != SK_S11_MAX) return 0;
    int e0 = hp->op0;
    *cpl = 0;
    if (hp->n_ops > e0 && hp->opcode[e0] == OP_CPL) { *cpl = 1; e0++; }
    const int nl = hp->n_ops - e0;
    if (nl < 1 || nl > QO_LAD_MAXN) return 0;
    const int op0 = hp->opcode[e0];
    if (op0 == OP_SER_LOSSY_L || op0 == OP_SER_L) *first = 0;
    else if (op0 == OP_SHUNT_LOSSY_C || op0 == OP_SHUNT_C) *first = 1;
    else return 0;
    int any_lossy = 0;
    for (int e = 0; e < nl; e++) {
        const int op = hp->opcode[e0 + e];
        const int series = ((e + *first) & 1) == 0;
        if (series ? !(op == OP_SER_LOSSY_L || op == OP_SER_L) : !(op == OP_SHUNT_LOSSY_C || op == OP_SHUNT_C)) return 0;
        if (op == OP_SER_LOSSY_L || op == OP_SHUNT_LOSSY_C) any_lossy = 1;
    }
    if (!any_lossy && !*cpl) return 0;    /* ideal ladders: the interpreter's imaginary-immittance path is cheaper */
    *n = nl;
    return 1;
}

/* The spot-frequency kernel (one thread per sample) serves reduce-only FP64 jobs on lumped cascades evaluated at a handful
 * of frequencies -- BASELINE config 3's harmonic-rejection yield at 2.4 / 4.8 / 7.2 GHz.  Any QO100NET_KERNEL override
 * but auto keeps jobs off it. */
static int spot_eligible(const DevProg *hp, int mode, int precision, int nf, const QoOverrides *ov, int *el0, int *nel)
{
    if (ov->kernel != QoOverrides::AUTO) return 0;
    if (mode != QO_MODE_REDUCE_ONLY || precision != 64 || hp->need_gd) return 0;
    if (nf > QO_SPOT_MAXF || hp->nspec < 1 || hp->nspec > QO_NSPEC_MAX) return 0;
    const int e0 = hp->op0, nl = hp->n_ops - e0;
    if (nl < 1 || nl > QO_SPOT_MAXEL) return 0;
    for (int e = 0; e < nl; e++) if (qo_tf_degree(hp->opcode[e0 + e]) < 0) return 0;
    for (int s = 0; s < hp->nspec; s++)
        if (hp->spec_kind[s] != SK_DEN2_MAX && hp->spec_kind[s] != SK_DEN2_MIN && hp->spec_kind[s] != SK_S11_MAX) return 0;
    *el0 = e0; *nel = nl;
    return 1;
}

/* Stability specs (SK_MU_MIN) need S11, S21, S12 and S22 of each point: only the interpreter and the compiled chain kernel form
 * them all.  The spot, transfer-function and ladder selectors refuse the spec kind; this gives qo_plan_tf_info and
 * qo_plan_analyze the reason. */
static const char *const qo_mu_reason = "stability spec needs all four S-parameters";
static int prog_has_mu(const DevProg *hp)
{
    for (int s = 0; s < hp->nspec; s++) if (hp->spec_kind[s] == SK_MU_MIN) return 1;
    return 0;
}

/* |S22| jobs on the polynomial and ladder kernels.  Every lumped branch and every lossless line is a symmetric, reciprocal two-port,
 * so S22 of a cascade N between (Rs, Rl) is exactly S11 of the reversed cascade between (Rl, Rs), and S21 is unchanged.  Each
 * element's draw depends on (sample, var) and its own parameters only, so the reversed job -- element e at n-1-e, terminations
 * swapped, |S22| specs turned into |S11| specs in the same order -- draws the same samples and runs on the |S11| instantiations
 * those kernels already have.  Builds the reversed network and program (rnet, rhp, rmask: the grid mask is the same) and returns
 * NULL when the spot, transfer-function or ladder kernel takes it (rtp, *rtf: its transfer-function analysis), else why not; the
 * job then runs on the interpreter or the compiled chain kernel, which evaluate S22 directly. */
static const char *s22_reversed(const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec, const qo_mc_cfg *cfg,
                                const DevProg *hp, int generic, const QoOverrides *ov, qo_net *rnet, DevProg *rhp,
                                std::vector<unsigned char> *rmask, TfPlan *rtp, int *rtf)
{
    const int mode = cfg ? cfg->mode : QO_MODE_FULL_S, precision = cfg && cfg->precision == 32 ? 32 : 64;
    if (generic || mode != QO_MODE_REDUCE_ONLY || precision != 64) return "not a reduce-only FP64 job on a lumped cascade";
    if (prog_has_mu(hp)) return qo_mu_reason;
    if (hp->need_s11) return "|S11| and |S22| specs in one job";
    /* a coupled line is symmetric too, but the kernels take it in front only; a measured block may be non-reciprocal */
    for (int e = 0; e < hp->n_ops; e++)
        if (qo_tf_degree(hp->opcode[e]) < 0 && hp->opcode[e] != OP_TLINE) return "|S22| needs a cascade of lumped branches and lines";
    const int n = net->n;
    memset(rnet, 0, sizeof *rnet);
    rnet->n = n; rnet->rs = net->rl; rnet->rl = net->rs;
    for (int e = 0; e < n; e++) rnet->e[e] = net->e[n - 1 - e];
    std::vector<qo_spec> rspec(spec, spec + nspec);
    for (qo_spec &s : rspec) if (s.kind == QO_SPEC_S22_MAX_DB) s.kind = QO_SPEC_S11_MAX_DB;
    std::vector<qo_tol> rtol;
    if (cfg->n_tol > 0) rtol.assign(cfg->tol, cfg->tol + cfg->n_tol);
    for (qo_tol &t : rtol) t.elem = n - 1 - t.elem;
    qo_mc_cfg rcfg = *cfg;
    rcfg.tol = rtol.data();
    int rgen = 0;
    double rfl = 0.0;
    if (build_prog(rnet, f, nf, rspec.data(), nspec, &rcfg, rhp, &rgen, &rfl, rmask) != QO_OK) return "reversed cascade does not compile";
    *rtf = qo_tf_plan_check(rhp, 1, precision, 0, f, nf, rmask->data(), ov, rtp);
    int a, b, c;
    if (*rtf || spot_eligible(rhp, mode, precision, nf, ov, &a, &b) || ladder_eligible(rhp, mode, precision, ov, &a, &b, &c)) return NULL;
    return rtp->reason;
}

/* the plan's kernel (QoKern, in order of precedence) */
static QoKern select_kernel(qo_plan *p, const double *f, int nf)
{
    const QoOverrides *ov = &p->ov;
    /* analysed for every plan: qo_plan_tf_info reports the result (or why it refused) whichever kernel runs */
    const int tf = qo_tf_plan_check(&p->hp, p->mode == QO_MODE_REDUCE_ONLY, p->precision, p->generic, f, nf, p->maskv.data(), ov, &p->tfp);
    if (!p->generic && p->mode == QO_MODE_REDUCE_ONLY && prog_has_mu(&p->hp)) { p->tfp.reason = qo_mu_reason; return K_LUMPED; }
    if (p->generic) return p->mode == QO_MODE_REDUCE_ONLY && nf <= QO_B_MAXNF && !ov->ustrip_item ? K_BOARD : K_GENERIC;
    if (spot_eligible(&p->hp, p->mode, p->precision, nf, ov, &p->spot_el0, &p->spot_nel)) return K_SPOT;
    if (tf) return K_TF;
    if (ladder_eligible(&p->hp, p->mode, p->precision, ov, &p->lad_n, &p->lad_first, &p->lad_cpl)) return K_LADDER;
    return K_LUMPED;
}

/* ---- plan ---------------------------------------------------------------- */
extern "C" void qo_plan_destroy(qo_plan *p)
{
    if (!p) return;
    for (int g = 0; g < p->ctx->ndev; g++) {
        cudaSetDevice(p->ctx->d[g].device);
        /* stream-ordered frees: back into the device's pool without a device-wide synchronisation */
        cudaStream_t st = p->ctx->d[g].stream;
        if (p->d[g].mem) cudaFreeAsync(p->d[g].mem, st);
        if (p->d[g].fs_mem) cudaFreeAsync(p->d[g].fs_mem, st);
    }
    if (p->pinned) cudaFreeHost(p->pinned);
    delete p;
}

/* angular frequency of grid point k; points past the grid (padding) repeat its last one */
static double grid_w(const double *f, int nf, size_t k) { return 6.283185307179586476925286766559 * f[k < (size_t)nf ? k : (size_t)nf - 1]; }

/* Measured two-port blocks: interpolate every block at every point (Qucs SPfile "linear"), convert to ABCD at the file's reference
 * impedance; blocks carry no tolerances, so this happens once per plan.  sblk: ABCD per (block, point) as four double2 (empty when
 * no element uses a block); sdet: the product of the blocks' determinants per point (empty when every block is reciprocal). */
static int block_tables(const qo_net *net, const double *f, int nf, int npts, std::vector<double2> *sblk, std::vector<double2> *sdet)
{
    int polar[QO_MAX_BLK];
    for (int b = 0; b < net->nblk; b++) polar[b] = 1;
    int used = 0;
    for (int e = 0; e < net->n; e++)
        if (net->e[e].kind == QO_SBLOCK) { polar[(int)net->e[e].p[0]] = net->e[e].p[1] != 0.0; used = 1; }
    if (!used) return QO_OK;
    int nonrecip = 0;
    sblk->resize((size_t)net->nblk * npts * 4);
    sdet->assign((size_t)npts, make_double2(1.0, 0.0));
    for (int b = 0; b < net->nblk; b++)
        for (int k = 0; k < npts; k++) {
            qo_c64 sv[4], m[4];
            qo_s2p_eval(net->blk[b], f[k < nf ? k : nf - 1], polar[b], sv);
            if (!qo_s_to_abcd(sv, net->blk[b]->z0, m)) {
                qo_set_error("S-parameter block %d has S21 = 0 at %g Hz: no chain matrix", b, f[k < nf ? k : nf - 1]);
                return QO_ERR_RANGE;
            }
            for (int q = 0; q < 4; q++) (*sblk)[((size_t)b * npts + k) * 4 + q] = make_double2(m[q].re, m[q].im);
            /* det(ABCD) = S12 / S21 */
            const double d = sv[1].re * sv[1].re + sv[1].im * sv[1].im;
            const double dr = (sv[2].re * sv[1].re + sv[2].im * sv[1].im) / d, di = (sv[2].im * sv[1].re - sv[2].re * sv[1].im) / d;
            if (fabs(dr - 1.0) > 1e-12 || fabs(di) > 1e-12) nonrecip = 1;
            const double2 o = (*sdet)[k];
            (*sdet)[k] = make_double2(o.x * dr - o.y * di, o.x * di + o.y * dr);
        }
    if (!nonrecip) sdet->clear();
    return QO_OK;
}

/* The coupler block in front of the ladder or transfer-function kernel.  Tables of sin/cos of its NOMINAL mode angles serve
 * every sample when each sample's angles stay within 0.1 rad of nominal over the whole grid (qo_ladder.cuh::lad_cpl_first); this
 * bounds that excursion up to wmax, the grid's largest angular frequency.  ke, ko: nominal even / odd mode angle per unit of w;
 * same: both modes alike, nominally and in tolerance. */
struct CplAngles { int fast, same; double ke, ko; };
static CplAngles cpl_angles(const DevProg *hp, double wmax, const QoOverrides *ov)
{
    CplAngles a = { 0, 0, 0.0, 0.0 };
    const int ec = hp->op0;                    /* the coupler op */
    double worst = 0;
    int ok = 1;
    if (hp->cplms_elem == ec) {
        /* physical element: bound the mode angles' excursion by running the analysis at every corner of the
         * tolerance box of the parameters it reads (<= 7 of them), plus 25 % margin for the interior */
        a.ke = hp->cplms_nom[2] / (360.0 * hp->nom[ec][4]); a.ko = hp->cplms_nom[3] / (360.0 * hp->nom[ec][4]);
        const int es = hp->cplms_sub;
        const int pe[7] = { ec, ec, es, es, es, ec, ec }, pk[7] = { 0, 1, 1, 2, 0, 3, 2 };      /* W S h t er ht L */
        double lo[7], hi[7];
        for (int q = 0; q < 7; q++) {
            const double nomv = hp->nom[pe[q]][pk[q]], t = hp->tvar[pe[q]][pk[q]] >= 0 ? fabs(hp->ttol[pe[q]][pk[q]]) : 0.0;
            const double dlt = hp->tmode[pe[q]][pk[q]] ? t : fabs(nomv) * t;
            lo[q] = nomv - dlt; hi[q] = nomv + dlt;
        }
        ok = !(hp->tvar[ec][4] >= 0);          /* a perturbed analysis frequency: not bounded here */
        for (int c = 0; c < 128 && ok; c++) {
            double v[7], o[4];
            for (int q = 0; q < 7; q++) v[q] = (c >> q) & 1 ? hi[q] : lo[q];
            if (!(v[0] > 0 && v[1] > 0 && v[2] > 0 && v[3] >= 0 && v[4] > 1 && v[5] > 0 && v[6] > 0)) { ok = 0; break; }
            qo_cpl_core(v[0], v[1], v[2], v[3], v[4], v[5], hp->nom[ec][4], v[6], o);
            const double de = fabs(o[2] / (360.0 * hp->nom[ec][4]) - a.ke), dn = fabs(o[3] / (360.0 * hp->nom[ec][4]) - a.ko);
            if (!(de == de) || !(dn == dn)) { ok = 0; break; }
            if (1.25 * de * wmax > worst) worst = 1.25 * de * wmax;
            if (1.25 * dn * wmax > worst) worst = 1.25 * dn * wmax;
        }
    } else {
        double lo[6], hi[6];
        for (int k = 0; k < 6; k++) {
            const double nomv = hp->nom[ec][k], t = hp->tvar[ec][k] >= 0 ? fabs(hp->ttol[ec][k]) : 0.0;
            const double dlt = hp->tmode[ec][k] ? t : fabs(nomv) * t;
            lo[k] = nomv - dlt; hi[k] = nomv + dlt;
        }
        ok = lo[4] > 0;
        for (int m = 0; m < 2 && ok; m++) {
            const double kn = hp->nom[ec][2 + m] / (360.0 * hp->nom[ec][4]);
            const double kmax = hi[2 + m] / (360.0 * lo[4]), kmin = lo[2 + m] / (360.0 * hi[4]);
            const double dk = fmax(kmax - kn, kn - kmin);
            if (dk * wmax > worst) worst = dk * wmax;
        }
        a.ke = hp->nom[ec][2] / (360.0 * hp->nom[ec][4]); a.ko = hp->nom[ec][3] / (360.0 * hp->nom[ec][4]);
        a.same = hp->nom[ec][2] == hp->nom[ec][3] && hp->tvar[ec][2] == hp->tvar[ec][3] && hp->ttol[ec][2] == hp->ttol[ec][3] &&
                 hp->tmode[ec][2] == hp->tmode[ec][3];
    }
    a.fast = ok && worst <= 0.1 && !ov->cpl_sincos;
    return a;
}

/* tables of the ladder and lumped kernels, in the plan's precision T, one entry per grid point, padded to a whole pair */
template <typename T>
static void chain_tables(qo_plan *p, const double *f, const std::vector<double2> &sblk, const std::vector<double2> &sdet, const CplAngles &ca)
{
    QoLayout &L = p->lay; QoTables &t = p->tab;
    const size_t npts = 2 * (size_t)p->npairs, tb = npts * sizeof(T);
    t.w2 = L.add(tb); t.wi2 = L.add(tb); t.m2 = L.add(npts);
    if (p->kern == K_LADDER) t.wsq2 = L.add(tb);
    if (p->kern == K_LADDER && p->cpl_fast) for (int c = 0; c < 4; c++) t.cpl[c] = L.add(tb);
    if (p->kern == K_LUMPED && !sblk.empty()) t.sblk = L.add(sblk.size() * sizeof(double2));
    if (p->kern == K_LUMPED && !sdet.empty()) t.sdet = L.add(sdet.size() * sizeof(double2));
    T *w2 = L.host<T>(t.w2), *wi2 = L.host<T>(t.wi2), *wsq2 = L.host<T>(t.wsq2), *cpl[4];
    for (int c = 0; c < 4; c++) cpl[c] = L.host<T>(t.cpl[c]);
    unsigned char *m2 = L.host<unsigned char>(t.m2);
    for (size_t k = 0; k < npts; k++) {
        const double w = grid_w(f, p->nf, k);
        w2[k] = (T)w; wi2[k] = (T)(1.0 / w); m2[k] = k < (size_t)p->nf ? p->maskv[k] : 0;
        if (wsq2) wsq2[k] = (T)(w * w);
        if (cpl[0]) { cpl[0][k] = (T)sin(ca.ke * w); cpl[1][k] = (T)cos(ca.ke * w); cpl[2][k] = (T)sin(ca.ko * w); cpl[3][k] = (T)cos(ca.ko * w); }
    }
    if (t.sblk != QO_NOTAB) memcpy(L.host<double2>(t.sblk), sblk.data(), sblk.size() * sizeof(double2));
    if (t.sdet != QO_NOTAB) memcpy(L.host<double2>(t.sdet), sdet.data(), sdet.size() * sizeof(double2));
}

/* tables of the transfer-function kernel, padded to whole iterations (padding repeats the last grid point and carries no spec
 * bit, so the loop needs no bounds checks) */
static void tf_tables(qo_plan *p, const double *f, const std::vector<double2> &sblk, const CplAngles &ca)
{
    QoLayout &L = p->lay; QoTables &t = p->tab;
    const int nf = p->nf, np = p->npairs;
    p->tf_pp = qo_tf_default_pp(&p->tfp, np);
    const int ppi = 32 * p->tf_pp;
    p->tf_niter = (np + ppi - 1) / ppi;
    /* + one iteration of padding: the kernel requests the next iteration's y values before it is done with the current one */
    const size_t npt = 2 * ((size_t)p->tf_niter + 1) * ppi, tb = npt * sizeof(double);
    /* a measured two-port in front: its row vector [1 Rs] M(f) per grid point rides in the four coupler-table slots */
    const bool front_blk = p->tfp.cpl_op >= 0 && p->tfp.front == 2;
    const bool front_s11 = front_blk && p->tfp.s11;         /* + its second row vector [1 -Rs] M for |S11| specs */
    t.yt = L.add(tb); t.xt = L.add(tb); t.wt = L.add(tb);
    if (p->cpl_fast || front_blk) for (int c = 0; c < 4; c++) t.cpl[c] = L.add(tb);
    if (front_s11) for (int c = 0; c < 4; c++) t.fu2[c] = L.add(tb);
    t.mb = L.add(2 * npt * sizeof(unsigned int));
    t.itm = L.add(((size_t)p->tf_niter * sizeof(uchar2) + 15) & ~(size_t)15);
    double *yt = L.host<double>(t.yt), *xt = L.host<double>(t.xt), *wt = L.host<double>(t.wt), *cpl[4], *fu2[4];
    for (int c = 0; c < 4; c++) { cpl[c] = L.host<double>(t.cpl[c]); fu2[c] = L.host<double>(t.fu2[c]); }
    unsigned int *mb = L.host<unsigned int>(t.mb); uchar2 *itm = L.host<uchar2>(t.itm);
    const double rs = p->hp.rs;
    for (size_t k = 0; k < npt; k++) {
        const size_t kc = k < (size_t)nf ? k : (size_t)nf - 1;
        const double w = grid_w(f, nf, k), x = w / p->tfp.wref;
        yt[k] = -(x * x); xt[k] = x; wt[k] = w;
        if (p->cpl_fast) { cpl[0][k] = sin(ca.ke * w); cpl[1][k] = cos(ca.ke * w); cpl[2][k] = sin(ca.ko * w); cpl[3][k] = cos(ca.ko * w); }
        if (front_blk) {
            const int blk = (int)p->hp.nom[p->tfp.cpl_op][0];
            const double2 *mm = &sblk[((size_t)blk * (size_t)(2 * np) + kc) * 4];
            cpl[0][k] = mm[0].x + rs * mm[2].x; cpl[1][k] = mm[0].y + rs * mm[2].y;
            cpl[2][k] = mm[1].x + rs * mm[3].x; cpl[3][k] = mm[1].y + rs * mm[3].y;
            if (front_s11) {
                fu2[0][k] = mm[0].x - rs * mm[2].x; fu2[1][k] = mm[0].y - rs * mm[2].y;
                fu2[2][k] = mm[1].x - rs * mm[3].x; fu2[3][k] = mm[1].y - rs * mm[3].y;
            }
        }
        unsigned int lo = 0, hi = 0;
        const unsigned char mk = k < (size_t)nf ? p->maskv[k] : 0;
        for (int sp = 0; sp < 4; sp++) {
            if ((mk >> sp) & 1u) lo |= 0xFFu << (8 * sp);
            if ((mk >> (sp + 4)) & 1u) hi |= 0xFFu << (8 * sp);
        }
        mb[2 * k] = lo; mb[2 * k + 1] = hi;
    }
    for (int it = 0; it < p->tf_niter; it++) {
        unsigned char any = 0, all = 0xFF;
        for (size_t k = (size_t)it * 2 * ppi; k < (size_t)(it + 1) * 2 * ppi; k++) {
            const unsigned char mk = k < (size_t)nf ? p->maskv[k] : 0;
            any |= mk; all &= mk;
        }
        itm[it] = make_uchar2(any, all);
    }
}

/* the tables the plan's kernel reads, in p->lay; where they lie, in p->tab */
static int build_tables(qo_plan *p, const qo_net *net, const double *f)
{
    QoLayout &L = p->lay; QoTables &t = p->tab;
    const int nf = p->nf, npts = 2 * p->npairs;
    t.prog = L.add(sizeof(DevProg));
    memcpy(L.host<DevProg>(t.prog), &p->hp, sizeof(DevProg));
    /* built for every plan with measured blocks; a transfer-function plan forms the row tables of its front block from them */
    std::vector<double2> sblk, sdet;
    const int rc = p->generic ? QO_OK : block_tables(net, f, nf, npts, &sblk, &sdet);
    if (rc) return rc;
    CplAngles ca = { 0, 0, 0.0, 0.0 };
    if ((p->kern == K_LADDER && p->lad_cpl) || (p->kern == K_TF && p->tfp.cpl_op >= 0 && p->tfp.front == 0)) {
        double wmax = 0;
        for (int k = 0; k < npts; k++) if (grid_w(f, nf, k) > wmax) wmax = grid_w(f, nf, k);
        ca = cpl_angles(&p->hp, wmax, &p->ov);
    }
    p->cpl_fast = ca.fast; p->cpl_same = ca.same;
    switch (p->kern) {
    case K_BOARD: case K_GENERIC:
        t.fgrid = L.add((size_t)nf * sizeof(double));
        memcpy(L.host<double>(t.fgrid), f, (size_t)nf * sizeof(double));
        t.mask = L.add((size_t)nf);
        memcpy(L.host<unsigned char>(t.mask), p->maskv.data(), (size_t)nf);
        break;
    case K_SPOT: break;                        /* its grid and spec bits travel in the kernel parameters */
    case K_TF: tf_tables(p, f, sblk, ca); break;
    case K_LADDER: case K_LUMPED:
        if (p->precision == 32) chain_tables<float>(p, f, sblk, sdet, ca);
        else chain_tables<double>(p, f, sblk, sdet, ca);
        break;
    }
    return QO_OK;
}

/* one allocation per device: the tables (one copy of p->lay), the counters (zeroed), the ticket area */
static int upload(qo_plan *p)
{
    const size_t cnt_bytes = (size_t)p->ncnt * sizeof(unsigned long long);
    p->tab.counters = align256(p->lay.buf.size());
    p->tab.ticket = align256(p->tab.counters + cnt_bytes);
    for (int g = 0; g < p->ctx->ndev; g++) {
        const DevCtx *dc = &p->ctx->d[g];
        CU(cudaSetDevice(dc->device));
        CU(cudaMallocAsync((void **)&p->d[g].mem, p->tab.ticket + QO_TICKET_BYTES, dc->stream));
        CU(cudaMemcpyAsync(p->d[g].mem, p->lay.buf.data(), p->lay.buf.size(), cudaMemcpyHostToDevice, dc->stream));
        CU(cudaMemsetAsync(p->counters(g), 0, cnt_bytes, dc->stream));
        CU(cudaStreamSynchronize(dc->stream));      /* a failed copy is reported by plan creation, not by the first launch */
    }
    return QO_OK;
}

static int plan_create(qo_ctx *ctx, const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec,
                       const qo_mc_cfg *cfg, const QoOverrides *ov, qo_plan **out)
{
    if (!ctx || !net || !f || nf <= 0 || !out || (nspec > 0 && !spec)) { qo_set_error("bad arguments"); return QO_ERR_ARG; }
    for (int k = 0; k < nf; k++)
        if (!(f[k] > 0.0) || !isfinite(f[k])) { qo_set_error("frequency %d is not a positive finite number", k); return QO_ERR_ARG; }
    qo_plan *p = new (std::nothrow) qo_plan();        /* value-initialised: what is not set here starts zeroed (QoTables: QO_NOTAB) */
    if (!p) return QO_ERR_NOMEM;
    p->ctx = ctx;
    p->ov = *ov;
    p->nf = nf;
    p->npairs = (nf + 1) / 2;
    p->precision = cfg && cfg->precision == 32 ? 32 : 64;
    p->mode = cfg ? cfg->mode : QO_MODE_FULL_S;
    int rc = build_prog(net, f, nf, spec, nspec, cfg, &p->hp, &p->generic, &p->flops_per_eval, &p->maskv);
    if (rc) { delete p; return rc; }
    if (p->generic && p->precision == 32) { delete p; qo_set_error("FP32 mode covers lumped/TL networks only"); return QO_ERR_UNSUPPORTED; }
    if (p->hp.need_gd && p->precision == 32) { delete p; qo_set_error("group-delay specs need FP64 (the 1e-6 relative frequency step is 8 float ulps)"); return QO_ERR_UNSUPPORTED; }
    if (p->generic)
        for (int e = 0; e < net->n; e++)
            if (net->e[e].kind == QO_SBLOCK) { qo_set_error("S-parameter blocks cannot be mixed with microstrip elements yet"); delete p; return QO_ERR_UNSUPPORTED; }
    p->ncnt = qo_ncnt(nspec, p->hp.hist_bins);
    p->f.assign(f, f + nf);
    const char *s22_why = NULL;
    qo_net *rnet = NULL;
    if (p->hp.need_s22) {
        rnet = new qo_net;
        DevProg *rhp = new DevProg;
        std::vector<unsigned char> rmask;
        TfPlan rtp;
        int rtf;
        s22_why = s22_reversed(net, f, nf, spec, nspec, cfg, &p->hp, p->generic, ov, rnet, rhp, &rmask, &rtp, &rtf);
        if (!s22_why) { p->hp = *rhp; p->maskv.swap(rmask); net = rnet; }
        delete rhp;
    }
    p->kern = select_kernel(p, f, nf);
    if (s22_why) p->tfp.reason = s22_why;
    p->kernel_name = qo_kern_name[p->kern];
    p->cj_debug = getenv("QO100NET_CHAIN_DEBUG") != NULL;
    rc = build_tables(p, net, f);
    delete rnet;
    if (rc == QO_OK) rc = upload(p);
    if (rc) { qo_plan_destroy(p); return rc; }
    if (p->kern == K_TF) tf_launch_setup(p, ov);
    *out = p;
    return QO_OK;
}

extern "C" int qo_plan_create(qo_ctx *ctx, const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec,
                              const qo_mc_cfg *cfg, qo_plan **out)
{
    qo_clear_error();
    QoOverrides ov;
    const int rc = qo_overrides_read(&ov);
    return rc ? rc : plan_create(ctx, net, f, nf, spec, nspec, cfg, &ov, out);
}

extern "C" int qo_plan_num_counters(const qo_plan *p) { return p ? p->ncnt : QO_ERR_ARG; }
extern "C" double qo_plan_flops_per_eval(const qo_plan *p) { return p ? p->flops_per_eval : 0.0; }
extern "C" int qo_plan_launches(const qo_plan *p) { return p ? p->launches : QO_ERR_ARG; }
/* Host-only (NVRTC compiles without a GPU): fold this job's element list into the chain kernel, compile it for sm_100a and report
 * what came out.  info[0] = compiled (0 also when libnvrtc is missing: qo_last_error says why), [1] = registers per thread,
 * [2] = spill bytes (-1 for either when NVRTC does not echo ptxas), [3] = cubin size in bytes. */
extern "C" int qo_chain_jit_analyze(const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec, const qo_mc_cfg *cfg, int info[4])
{
    qo_clear_error();
    if (!net || !f || nf <= 0 || !cfg || !info || (nspec > 0 && !spec)) return QO_ERR_ARG;
    for (int i = 0; i < 4; i++) info[i] = 0;
    QoOverrides ov;                          /* nothing here depends on them, but a bad value is refused as everywhere else */
    int rc = qo_overrides_read(&ov);
    if (rc) return rc;
    DevProg hp;
    int generic = 0;
    double flops = 0.0;
    std::vector<unsigned char> maskv;
    rc = build_prog(net, f, nf, spec, nspec, cfg, &hp, &generic, &flops, &maskv);
    if (rc) return rc;
    if (generic) { qo_set_error("microstrip networks run on their own kernels"); return QO_ERR_UNSUPPORTED; }
    const std::string src = qcj_source(&hp, cfg->mode == QO_MODE_FULL_S);
    const QcjEntry *e = qcj_get(src, qcj_hash(src), true, getenv("QO100NET_CHAIN_DEBUG") != NULL, false);
    info[0] = e->ok; info[1] = e->regs; info[2] = e->spill_bytes; info[3] = e->cubin_bytes;
    if (!e->ok) qo_set_error("%s", e->log.substr(0, 600).c_str());
    return QO_OK;
}

extern "C" const char *qo_plan_kernel_name(const qo_plan *p) { return p ? p->kernel_name : ""; }
extern "C" const char *qo_plan_tf_info(const qo_plan *p, int info[6], double *self_check_err, unsigned int *fused, double *fused_err)
{
    if (!p) return "";
    if (info) { info[0] = p->kern == K_TF; info[1] = p->tfp.nn; info[2] = p->tfp.den; info[3] = p->tfp.kn; info[4] = p->tfp.kd; info[5] = p->tfp.deg; }
    if (self_check_err) *self_check_err = p->tfp.err;
    if (fused) *fused = p->tfp.fused;
    if (fused_err) *fused_err = p->tfp.fused_err;
    return p->tfp.reason ? p->tfp.reason : "";
}
extern "C" uint64_t qo_plan_h2d_bytes(const qo_plan *p) { return p ? p->lay.buf.size() : 0; }

/* host-only part of qo_plan_create: compile the network, decide about the transfer-function kernel (needs no GPU).
 * Returns the reason (or the error), *sel = 1 when the job takes the transfer-function kernel, < 0 on an error */
static const char *plan_analyze(const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec, const qo_mc_cfg *cfg,
                                TfPlan *tp, int *sel, double *seconds)
{
    qo_clear_error();
    memset(tp, 0, sizeof *tp);
    *sel = 0;
    if (!net || !f || nf <= 0) { *sel = QO_ERR_ARG; return "bad arguments"; }
    QoOverrides ov;
    if ((*sel = qo_overrides_read(&ov)) != QO_OK) return qo_last_error();
    DevProg *hp = new DevProg;
    int generic = 0;
    double fl = 0;
    std::vector<unsigned char> maskv;
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    int rc = build_prog(net, f, nf, spec, nspec, cfg, hp, &generic, &fl, &maskv);
    const char *reason = "network does not compile";
    if (rc == QO_OK) {
        const int precision = cfg && cfg->precision == 32 ? 32 : 64;
        const int mode = cfg ? cfg->mode : QO_MODE_FULL_S;
        *sel = qo_tf_plan_check(hp, mode == QO_MODE_REDUCE_ONLY, precision, generic, f, nf, maskv.data(), &ov, tp);
        if (!generic && mode == QO_MODE_REDUCE_ONLY && prog_has_mu(hp)) { *sel = 0; tp->reason = qo_mu_reason; }
        if (hp->need_s22) {             /* the analysis of the program that runs: the reversed cascade's when it is taken */
            qo_net *rnet = new qo_net;
            DevProg *rhp = new DevProg;
            std::vector<unsigned char> rmask;
            TfPlan *rtp = new TfPlan;
            int rtf = 0;
            const char *why = s22_reversed(net, f, nf, spec, nspec, cfg, hp, generic, &ov, rnet, rhp, &rmask, rtp, &rtf);
            if (why) tp->reason = why;
            else { *tp = *rtp; *sel = rtf; }
            delete rtp; delete rhp; delete rnet;
        }
        reason = tp->reason ? tp->reason : "";
    }
    clock_gettime(CLOCK_MONOTONIC, &t1);
    if (seconds) *seconds = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
    delete hp;
    return reason;
}

extern "C" const char *qo_plan_analyze(const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec, const qo_mc_cfg *cfg,
                                       int info[6], double *self_check_err, unsigned int *fused, double *fused_err, double *seconds)
{
    if (!net || !f || nf <= 0 || !info) return "bad arguments";
    TfPlan tp;
    const char *reason = plan_analyze(net, f, nf, spec, nspec, cfg, &tp, &info[0], seconds);
    if (info[0] < 0) return reason;
    info[1] = tp.nn; info[2] = tp.den; info[3] = tp.kn; info[4] = tp.kd; info[5] = tp.deg;
    if (self_check_err) *self_check_err = tp.err;
    if (fused) *fused = tp.fused;
    if (fused_err) *fused_err = tp.fused_err;
    return reason;
}

#define QO_TS_RUN_INTS 7
/* the thread-per-sample kernel's run table, QO_TS_RUN_INTS ints per run (first group, groups, spec bits seen by some point, by
 * every point, numerator pairs, E coefficients, fused-margin coefficients); returns the number of runs (0 when the job cannot run
 * thread-per-sample), meta = { plain runs (the fused spec's follow), points per group } */
static int ts_runs_out(const TfPlan *tp, int *runs, int cap, int meta[2])
{
    if (!tp->ts_runs_ok) { if (meta) meta[0] = meta[1] = 0; return 0; }
    if (meta) { meta[0] = tp->ts_nplain; meta[1] = qo_ts_group_points(tp); }
    for (int r = 0; r < tp->ts_nruns && r < cap; r++) {
        const TsRun &u = tp->runs[r];
        int *o = runs + QO_TS_RUN_INTS * r;
        o[0] = u.g0; o[1] = u.ngroups; o[2] = (int)u.any; o[3] = (int)u.all; o[4] = u.kn; o[5] = u.ke; o[6] = u.kf;
    }
    return tp->ts_nruns;
}

extern "C" int qo_plan_ts_runs(const qo_plan *p, int *runs, int cap, int meta[2])
{
    if (!p || (cap > 0 && !runs)) return QO_ERR_ARG;
    return ts_runs_out(&p->tfp, runs, cap, meta);
}

extern "C" int qo_plan_analyze_ts_runs(const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec, const qo_mc_cfg *cfg,
                                       int *runs, int cap, int meta[2])
{
    if (cap > 0 && !runs) return QO_ERR_ARG;
    TfPlan tp;
    int sel;
    plan_analyze(net, f, nf, spec, nspec, cfg, &tp, &sel, NULL);
    if (sel < 0) return sel;
    return ts_runs_out(&tp, runs, cap, meta);
}

/* the histogram screen of the thread-per-sample kernel: "ok" or why the plan declined it; info = { eps, smallest and largest
 * threshold covered, worst error bound over eps/8 }; meta = { seed runs (the first ones of the run table), screened runs,
 * whether the plan's last thread-per-sample launch ran qo_mc_ts_screen_kernel (0 before a launch and for the analyze form) } */
static const char *ts_screen_out(const TfPlan *tp, double info[4], int meta[3])
{
    int n = 0;
    for (int r = 0; r < tp->ts_nplain && tp->ts_screen_reason && !strcmp(tp->ts_screen_reason, "ok"); r++) n += tp->runs[r].kf > 0;
    if (info) { info[0] = tp->ts_screen_eps; info[1] = tp->ts_screen_mlo; info[2] = tp->ts_screen_mhi; info[3] = tp->ts_screen_bound; }
    if (meta) { meta[0] = tp->ts_nseed; meta[1] = n; meta[2] = 0; }
    return tp->ts_screen_reason ? tp->ts_screen_reason : tp->reason && strcmp(tp->reason, "ok") ? tp->reason : "the job does not run thread-per-sample";
}

extern "C" const char *qo_plan_ts_screen(const qo_plan *p, double info[4], int meta[3])
{
    if (!p) return "";
    const char *r = ts_screen_out(&p->tfp, info, meta);
    if (meta) meta[2] = p->ts_screen_ran;
    return r;
}

extern "C" const char *qo_plan_analyze_ts_screen(const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec, const qo_mc_cfg *cfg,
                                                 double info[4], int meta[3])
{
    TfPlan tp;
    int sel;
    const char *reason = plan_analyze(net, f, nf, spec, nspec, cfg, &tp, &sel, NULL);
    if (sel < 0) { if (meta) meta[0] = meta[1] = meta[2] = sel; return reason; }
    return ts_screen_out(&tp, info, meta);
}

extern "C" int qo_plan_reset(qo_plan *p)
{
    if (!p) return QO_ERR_ARG;
    for (int g = 0; g < p->ctx->ndev; g++) {
        CU(cudaSetDevice(p->ctx->d[g].device));
        CU(cudaMemsetAsync(p->counters(g), 0, (size_t)p->ncnt * sizeof(unsigned long long), p->ctx->d[g].stream));
    }
    return QO_OK;
}

/* Pre-pass of the physical coupled-line element: one thread per sample turns that sample's geometry / substrate
 * draws (same Philox stream, same variables as every other kernel) into Z0e, Z0o, theta_e, theta_o with the
 * coupled-microstrip analysis (qo_cpl_core.h) -- ~150 pow/exp/log per SAMPLE, done here at full lane
 * efficiency instead of by one lane of the warp that owns the sample. */
__global__ void qo_cplms_kernel(const DevProg *__restrict__ prog, unsigned long long sample_offset, unsigned long long n, double *__restrict__ out)
{
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int ec = prog->cplms_elem, es = prog->cplms_sub;
    double pc[6], ps[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        pc[k] = prog->nom[ec][k];
        int tv = prog->tvar[ec][k];
        if (tv >= 0) pc[k] = qo_stream_apply(pc[k], prog->ttol[ec][k], qo_stream_variate(prog->seed, sample_offset + i, (uint32_t)tv, prog->dist), prog->tmode[ec][k]);
        ps[k] = prog->nom[es][k];
        tv = prog->tvar[es][k];
        if (tv >= 0) ps[k] = qo_stream_apply(ps[k], prog->ttol[es][k], qo_stream_variate(prog->seed, sample_offset + i, (uint32_t)tv, prog->dist), prog->tmode[es][k]);
    }
    double o[4];
    qo_cpl_core(pc[0], pc[1], ps[1], ps[2], ps[0], pc[3], pc[4], pc[2], o);
    out[4 * i + 0] = o[0]; out[4 * i + 1] = o[1]; out[4 * i + 2] = o[2]; out[4 * i + 3] = o[3];
}

template <typename T>
static int launch_lumped(qo_plan *p, int g, unsigned long long off, unsigned long long n, unsigned long long *cnt, QoPlanes pl, int full_s)
{
    DevCtx *dc = &p->ctx->d[g];
    typedef typename QoVec2<T>::type V2;
    const DevProg *prog = p->dev<DevProg>(g, p->tab.prog);
    const V2 *w2 = p->dev<V2>(g, p->tab.w2), *wi2 = p->dev<V2>(g, p->tab.wi2); const uchar2 *m2 = p->dev<uchar2>(g, p->tab.m2);
    const int resident = dc->sm_count * 2;                  /* __launch_bounds__(256, 2) */
    const unsigned long long warps_resident = (unsigned long long)resident * QO_WARPS;
    /* split the frequency axis only when there are too few samples to fill the GPU (sweeps) */
    int nchunks = 1, ppc = p->npairs;
    if (full_s && n < warps_resident) {
        unsigned long long want = (warps_resident + n - 1) / n;
        int maxc = (p->npairs + 31) / 32;
        nchunks = (int)(want < (unsigned long long)maxc ? want : (unsigned long long)maxc);
        if (nchunks < 1) nchunks = 1;
        ppc = ((p->npairs + nchunks - 1) / nchunks + 31) / 32 * 32;
        nchunks = (p->npairs + ppc - 1) / ppc;
    }
    unsigned long long units = n * (unsigned long long)nchunks;
    unsigned long long blocks = (units + QO_WARPS - 1) / QO_WARPS;
    int grid = (int)(blocks < (unsigned long long)resident ? blocks : (unsigned long long)resident);
    if (grid < 1) grid = 1;
    if (sizeof(T) == sizeof(double) && p->ov.chain >= 0 && !p->cj_failed[full_s ? 1 : 0]) {
        /* large jobs: the element list compiled into the kernel (qo_chain_jit.h) */
        const int fs = full_s ? 1 : 0;
        const unsigned long long evals = n * (unsigned long long)p->nf;
        const QcjEntry *je = (const QcjEntry *)p->cj[fs];
        if (!je && (p->ov.chain == 1 || evals >= QO_CJ_MIN_CACHED)) {
            if (p->cj_src[fs].empty()) { p->cj_src[fs] = qcj_source(&p->hp, fs); p->cj_hash[fs] = qcj_hash(p->cj_src[fs]); }
            je = qcj_get(p->cj_src[fs], p->cj_hash[fs], p->ov.chain == 1 || evals >= QO_CJ_MIN_EVALS, p->cj_debug != 0);
            if (je && !je->ok) {
                p->cj_failed[fs] = 1;
                if (p->ov.chain == 1) { qo_set_error("QO100NET_CHAIN=jit: %s", je->log.substr(0, 400).c_str()); return QO_ERR_UNSUPPORTED; }
                je = NULL;
            }
            p->cj[fs] = je;
        }
        if (je) {
            if (je->blocks_per_sm > 2) {        /* built for more resident blocks than the interpreter's two: size the persistent grid accordingly */
                const int res2 = dc->sm_count * je->blocks_per_sm;
                grid = (int)(blocks < (unsigned long long)res2 ? blocks : (unsigned long long)res2);
                if (grid < 1) grid = 1;
            }
            int a_nf = p->nf, a_np = p->npairs;
            void *args[] = { &prog, &w2, &wi2, &m2, &a_nf, &a_np, &ppc, &nchunks, &off, &n, &cnt, &pl };
            CU(cudaLaunchKernel((const void *)je->kern, dim3((unsigned)grid), dim3(QO_TPB), args, 0, dc->stream));
            p->kernel_name = "qo_mc_chain_jit_kernel";
            return QO_OK;
        }
    }
    p->kernel_name = "qo_mc_lumped_kernel";
#define QO_LAUNCH(FS, TR, GD, S22, MU)                                                                              \
    qo_mc_lumped_kernel<T, FS, TR, GD, S22, MU><<<grid, QO_TPB, 0, dc->stream>>>(prog, w2, wi2, m2, p->nf, p->npairs, ppc, nchunks, off, n, cnt, pl)
#define QO_LAUNCH_TR(FS, GD, S22) do { if (p->hp.has_trig) QO_LAUNCH(FS, true, GD, S22, false); else QO_LAUNCH(FS, false, GD, S22, false); } while (0)
    /* |S22| and stability jobs have instantiations of their own: the others' machine code stays as it was.  A stability job is
     * FP64 and has a measured block, hence TRIG, and never group delay (build_prog); its one instantiation serves |S22| too. */
    if (full_s) QO_LAUNCH_TR(true, false, false);
    else if (prog_has_mu(&p->hp)) { if constexpr (sizeof(T) == sizeof(double)) QO_LAUNCH(false, true, false, true, true); }
    else if (p->hp.need_s22) { if (p->hp.need_gd) QO_LAUNCH_TR(false, true, true); else QO_LAUNCH_TR(false, false, true); }
    else if (p->hp.need_gd) QO_LAUNCH_TR(false, true, false);
    else QO_LAUNCH_TR(false, false, false);
#undef QO_LAUNCH_TR
#undef QO_LAUNCH
    CU(cudaGetLastError());
    return QO_OK;
}

static int launch_ladder(qo_plan *p, int g, unsigned long long off, unsigned long long n, unsigned long long *cnt, const double *cplms)
{
    DevCtx *dc = &p->ctx->d[g];
    const DevProg *hp = &p->hp;
    const QoTables &t = p->tab;
    LadParams P;
    memset(&P, 0, sizeof P);
    P.prog = p->dev<DevProg>(g, t.prog);
    P.wt = p->dev<void>(g, t.w2); P.wit = p->dev<void>(g, t.wi2); P.wsqt = p->dev<void>(g, t.wsq2); P.m2 = p->dev<uchar2>(g, t.m2);
    P.counters = cnt;
    P.cse = p->dev<void>(g, t.cpl[0]); P.cce = p->dev<void>(g, t.cpl[1]); P.cso = p->dev<void>(g, t.cpl[2]); P.cco = p->dev<void>(g, t.cpl[3]);
    P.cpl_fast = p->cpl_fast; P.cpl_same = p->cpl_same;
    P.cplms = cplms; P.op0 = hp->op0;
    P.ticket = p->ticket(g);
    CU(cudaMemsetAsync(P.ticket, 0, sizeof(unsigned long long), dc->stream));
    P.sample_offset = off; P.nsamples = n; P.seed = hp->seed;
    P.rs = hp->rs; P.rl = hp->rl; P.k21 = hp->k21; P.hist_lo = hp->hist_lo; P.hist_hi = hp->hist_hi;
    for (int s = 0; s < QO_LAD_NSPEC; s++) {
        const int neg = s < hp->nspec && hp->spec_kind[s] == SK_DEN2_MIN;
        P.neg[s] = neg;
        P.thr[s] = s < hp->nspec ? (neg ? -hp->spec_thr[s] : hp->spec_thr[s]) : 0.0;
        P.is_s11[s] = s < hp->nspec && hp->spec_kind[s] == SK_S11_MAX;
    }
    P.npairs = p->npairs; P.n_var = hp->n_var; P.n_ops = hp->n_ops; P.nspec = hp->nspec; P.dist = hp->dist;
    P.hist_bins = hp->hist_bins;
    P.hist_spec = hp->hist_bins > 0 ? hp->hist_spec : -1;
    P.hist_kind = hp->hist_bins > 0 ? hp->spec_kind[hp->hist_spec] : 0;
    int rc = qo_ladder_launch(p->lad_n, p->lad_first, p->lad_cpl, hp->need_s11 ? 2 : 1, p->precision, dc->sm_count, &P, dc->stream);
    if (rc < 0) { qo_set_error("no ladder kernel instantiation for n=%d first=%d cpl=%d", p->lad_n, p->lad_first, p->lad_cpl); return QO_ERR_UNSUPPORTED; }
    if (rc) { qo_set_error("ladder kernel launch: %s", cudaGetErrorString((cudaError_t)rc)); return QO_ERR_CUDA; }
    return QO_OK;
}

/* what launch_tf needs beyond the tables, decided once per plan: the coupler block's form (matched source, uniformly spaced
 * grid) and whether large launches may run thread-per-sample (on the run table the analysis built: qo_tf.cu::tf_ts_runs) */
static void tf_launch_setup(qo_plan *p, const QoOverrides *ov)
{
    const DevProg *hp = &p->hp;
    const int cop = p->tfp.cpl_op;
    const int front = cop >= 0 ? p->tfp.front : 0;
    /* source resistance == the coupler's (unperturbed) reference impedance: the block's row vector collapses (qo_tf.cuh::tf_cpl_matched) */
    p->tf_cpl_matched = cop >= 0 && !front && !p->tfp.s11 && hp->tvar[cop][5] < 0 && hp->nom[cop][5] == hp->rs;
    /* uniformly spaced grid (config 5: linear 70 MHz .. 4 GHz): the coupler's mode angles advance by a constant per iteration */
    p->tf_cpl_lin = 0; p->tf_cpl_dw1 = 0.0;
    if (cop >= 0 && !front && !p->tfp.s11 && p->nf >= 3) {
        const double d0 = p->f[1] - p->f[0];
        int lin = d0 > 0.0;
        for (int k = 2; k < p->nf && lin; k++) if (fabs((p->f[k] - p->f[k - 1]) - d0) > 1e-9 * fabs(d0)) lin = 0;
        if (lin) { p->tf_cpl_lin = 1; p->tf_cpl_dw1 = 6.283185307179586476925286766559 * ((p->f[p->nf - 1] - p->f[0]) / (double)(p->nf - 1)); }
    }
    const bool rot_same = p->tf_cpl_lin && p->tf_cpl_matched && p->cpl_same && hp->cplms_elem < 0;
    p->ts_ok = ov->kernel != QoOverrides::TF && qo_ts_eligible(&p->tfp, hp->nspec, rot_same);     /* KERNEL=tf: warp-per-sample only (A/B runs) */
}

static int launch_tf(qo_plan *p, int g, unsigned long long off, unsigned long long n, unsigned long long *cnt, const double *cplms)
{
    DevCtx *dc = &p->ctx->d[g];
    const DevProg *hp = &p->hp;
    const QoTables &t = p->tab;
    TfParams P;
    memset(&P, 0, sizeof P);
    P.prog = p->dev<DevProg>(g, t.prog);
    P.yt = p->dev<double2>(g, t.yt); P.xt = p->dev<double2>(g, t.xt); P.wt = p->dev<double2>(g, t.wt);
    P.mb = p->dev<uint4>(g, t.mb); P.itm = p->dev<uchar2>(g, t.itm);
    P.cse = p->dev<double2>(g, t.cpl[0]); P.cce = p->dev<double2>(g, t.cpl[1]); P.cso = p->dev<double2>(g, t.cpl[2]); P.cco = p->dev<double2>(g, t.cpl[3]);
    P.cpl_fast = p->cpl_fast; P.cpl_same = p->cpl_same; P.cpl_op = p->tfp.cpl_op;
    /* source resistance == the coupler's (unperturbed) reference impedance: the block's row vector collapses (qo_tf.cuh::tf_cpl_matched) */
    P.front = p->tfp.cpl_op >= 0 ? p->tfp.front : 0;
    for (int c = 0; c < 4; c++) P.fu2[c] = p->dev<double2>(g, t.fu2[c]);
    P.cpl_matched = p->tf_cpl_matched;
    P.cpl_lin = p->tf_cpl_lin; P.cpl_dw = p->tf_cpl_dw1 * (double)(64 * p->tf_pp);
    P.cplms = cplms;
    P.counters = cnt; P.ticket = p->ticket(g);
    CU(cudaMemsetAsync(P.ticket, 0, QO_TICKET_BYTES, dc->stream));
    P.sample_offset = off; P.nsamples = n; P.seed = hp->seed;
    P.rs = hp->rs; P.rl = hp->rl; P.k21 = hp->k21; P.hist_lo = hp->hist_lo; P.hist_hi = hp->hist_hi;
    P.wref = p->tfp.wref; P.zn = sqrt(hp->rs * hp->rl); P.zni = 1.0 / P.zn;
    for (int s = 0; s < QO_TF_NSPEC; s++) {
        P.neg[s] = s < hp->nspec && hp->spec_kind[s] == SK_DEN2_MIN;
        P.s11[s] = s < hp->nspec && hp->spec_kind[s] == SK_S11_MAX;
        P.gd[s] = s < hp->nspec && hp->spec_kind[s] == SK_GD_MAX;
        P.thr[s] = s < hp->nspec ? (P.gd[s] ? hp->spec_thr[s] * p->tfp.wref : hp->spec_thr[s]) : 0.0;
    }
    P.niter = p->tf_niter; P.n_var = hp->n_var; P.n_el = p->tfp.n_el; P.el0 = p->tfp.el0; P.kn = p->tfp.kn; P.kd = p->tfp.kd; P.den = p->tfp.den; P.nspec = hp->nspec; P.dist = hp->dist;
    P.hist_bins = hp->hist_bins;
    P.hist_spec = hp->hist_bins > 0 ? hp->hist_spec : -1;
    /* the bulk of a large launch runs thread-per-sample (qo_ts.cuh): whole rounds of one sample per resident thread, dealt
     * statically; what is left over (less than one wave) stays on the warp-per-sample kernel below */
    if (p->ts_ok && p->tfp.ts_runs_ok) {
        /* worth it from a few batches per resident warp on (one wave = every resident thread one sample) */
        const unsigned long long wave = (unsigned long long)qo_ts_wave_threads(&p->tfp, dc->sm_count);
        const unsigned long long nb = wave && n >= 2 * wave ? n / 32ull : 0;
        if (nb > 0) {
            TsParams Q;
            memset(&Q, 0, sizeof Q);
            Q.t = P;
            Q.t.nsamples = nb * 32ull;
            Q.y1 = p->dev<double>(g, t.yt); Q.x1 = p->dev<double>(g, t.xt); Q.mw = p->dev<uint2>(g, t.mb);
            Q.npt = p->tfp.ts_npt;
            Q.nruns = p->tfp.ts_nruns; Q.nplain = p->tfp.ts_nplain;
            memcpy(Q.runs, p->tfp.runs, sizeof Q.runs);
            Q.nbatches = nb;
            Q.ticket = P.ticket + 1;
            Q.w0 = 6.283185307179586476925286766559 * p->f[0];
            Q.dw = p->nf > 1 ? 6.283185307179586476925286766559 * ((p->f[p->nf - 1] - p->f[0]) / (double)(p->nf - 1)) : 0.0;
            Q.screen_eps = p->tfp.ts_screen_eps; Q.screen_mlo = p->tfp.ts_screen_mlo; Q.screen_mhi = p->tfp.ts_screen_mhi;
            int rts = qo_ts_launch(&p->tfp, dc->sm_count, &Q, dc->stream);
            if (rts) { qo_set_error("thread-per-sample kernel launch: %s", cudaGetErrorString((cudaError_t)rts)); return QO_ERR_CUDA; }
            p->kernel_name = "qo_mc_ts_kernel";                   /* the family: qo_plan_ts_screen says whether its screen flavour ran */
            p->ts_screen_ran = p->tfp.ts_nseed > 0;
            p->launches++;
            off += nb * 32ull; n -= nb * 32ull;
            if (n == 0) return QO_OK;
            P.sample_offset = off; P.nsamples = n;
        }
    }
    int rc = qo_tf_launch(&p->tfp, p->tf_pp, dc->sm_count, &P, dc->stream);
    if (rc < 0) { qo_set_error("no transfer-function kernel instantiation for nn=%d den=%d pp=%d", p->tfp.nn, p->tfp.den, p->tf_pp); return QO_ERR_UNSUPPORTED; }
    if (rc) { qo_set_error("transfer-function kernel launch: %s", cudaGetErrorString((cudaError_t)rc)); return QO_ERR_CUDA; }
    return QO_OK;
}

static int launch_spot(qo_plan *p, int g, unsigned long long off, unsigned long long n, unsigned long long *cnt)
{
    DevCtx *dc = &p->ctx->d[g];
    const DevProg *hp = &p->hp;
    SpotParams P;
    memset(&P, 0, sizeof P);
    P.prog = p->dev<DevProg>(g, p->tab.prog); P.counters = cnt;
    P.sample_offset = off; P.nsamples = n; P.seed = hp->seed;
    P.rs = hp->rs; P.rl = hp->rl; P.k21 = hp->k21; P.hist_lo = hp->hist_lo; P.hist_hi = hp->hist_hi;
    for (int k = 0; k < p->nf; k++) { P.w[k] = grid_w(p->f.data(), p->nf, k); P.mask[k] = p->maskv[k]; }
    for (int s = 0; s < hp->nspec; s++) { P.thr[s] = hp->spec_thr[s]; P.kind[s] = hp->spec_kind[s]; }
    P.nf = p->nf; P.n_el = p->spot_nel; P.el0 = p->spot_el0; P.nspec = hp->nspec; P.dist = hp->dist;
    P.hist_bins = hp->hist_bins;
    P.hist_spec = hp->hist_bins > 0 ? hp->hist_spec : -1;
    int rc = qo_spot_launch(hp->need_s11, dc->sm_count, &P, dc->stream);
    if (rc) { qo_set_error("spot kernel launch: %s", cudaGetErrorString((cudaError_t)rc)); return QO_ERR_CUDA; }
    return QO_OK;
}

/* FULL_S launches with enough samples to fill the GPU go through the transfer-function kernel's FULL_S flavour when the
 * job allows it.  The analysis runs once, at the first such launch (nominal sweeps -- one sample -- never pay for it). */
#define QO_FS_TF_MIN_SAMPLES 1024
static int launch_tf_fs(qo_plan *p, int g, unsigned long long off, unsigned long long n, QoPlanes pl)
{
    DevCtx *dc = &p->ctx->d[g];
    DevPlan *d = &p->d[g];
    const DevProg *hp = &p->hp;
    QoLayout &L = p->fs_lay;
    if (L.buf.empty()) {
        const int ppi = 32 * 2;
        p->fs_niter = (p->npairs + ppi - 1) / ppi;
        const size_t npt = 2 * (size_t)p->fs_niter * ppi;
        p->fs_yt = L.add(npt * sizeof(double)); p->fs_xt = L.add(npt * sizeof(double));
        double *yt = L.host<double>(p->fs_yt), *xt = L.host<double>(p->fs_xt);
        for (size_t k = 0; k < npt; k++) {
            const double x = grid_w(p->f.data(), p->nf, k) / p->fsp.wref;
            yt[k] = -(x * x); xt[k] = x;
        }
    }
    if (!d->fs_mem) {
        CU(cudaMallocAsync((void **)&d->fs_mem, L.buf.size(), dc->stream));
        CU(cudaMemcpyAsync(d->fs_mem, L.buf.data(), L.buf.size(), cudaMemcpyHostToDevice, dc->stream));
        CU(cudaStreamSynchronize(dc->stream));
    }
    TfFsParams P;
    memset(&P, 0, sizeof P);
    P.prog = p->dev<DevProg>(g, p->tab.prog); P.yt = (const double2 *)(d->fs_mem + p->fs_yt); P.xt = (const double2 *)(d->fs_mem + p->fs_xt);
    P.s11 = pl.s11; P.s21 = pl.s21; P.s12 = pl.s12; P.s22 = pl.s22;
    P.planes_al32 = ((((size_t)pl.s11) | ((size_t)pl.s21) | ((size_t)pl.s12) | ((size_t)pl.s22)) & 31) == 0;
    P.ticket = p->ticket(g);
    CU(cudaMemsetAsync(P.ticket, 0, sizeof(unsigned long long), dc->stream));
    P.sample_offset = off; P.nsamples = n; P.seed = hp->seed;
    P.rs = hp->rs; P.rl = hp->rl; P.k21 = hp->k21; P.wref = p->fsp.wref; P.zn = sqrt(hp->rs * hp->rl); P.zni = 1.0 / P.zn;
    P.nf = p->nf; P.niter = p->fs_niter; P.kn = p->fsp.kn; P.kd = p->fsp.kd; P.n_var = hp->n_var; P.n_el = p->fsp.n_el; P.el0 = p->fsp.el0; P.dist = hp->dist;
    int dmode = p->fsp.den == QO_TF_DEN_NONE ? 0 : p->fsp.den == QO_TF_DEN_D ? 1 : 2;
    if (dmode == 2) {
        for (int e = 0; e < p->fsp.n_el; e++) {
            const int op = hp->opcode[p->fsp.el0 + e];
            if (!(op == OP_SER_R || op == OP_SER_L || op == OP_SHUNT_C)) P.fac[P.nfac++] = (unsigned char)e;
        }
    }
    int rc = qo_tf_fs_launch(dmode, dc->sm_count, &P, dc->stream);
    if (rc) { qo_set_error("FULL_S transfer-function kernel launch: %s", cudaGetErrorString((cudaError_t)rc)); return QO_ERR_CUDA; }
    return QO_OK;
}

static int launch_generic(qo_plan *p, int g, unsigned long long off, unsigned long long n, unsigned long long *cnt, QoPlanes pl, int full_s)
{
    DevCtx *dc = &p->ctx->d[g];
    const DevProg *prog = p->dev<DevProg>(g, p->tab.prog);
    const double *fgrid = p->dev<double>(g, p->tab.fgrid); const unsigned char *mask = p->dev<unsigned char>(g, p->tab.mask);
    if (p->kern == K_BOARD) {
        /* yield at a handful of frequencies: one thread per board, the frequencies side by side (qo_ustrip_board.cuh) */
        const unsigned long long cap = (unsigned long long)dc->sm_count * QO_B_MINB, want = (n + QO_B_TPB - 1) / QO_B_TPB;
        const int grid = (int)(want < cap ? want : cap);
        switch (p->nf) {
        case 1: qo_mc_board_kernel<1><<<grid, QO_B_TPB, 0, dc->stream>>>(prog, fgrid, mask, off, n, cnt); break;
        case 2: qo_mc_board_kernel<2><<<grid, QO_B_TPB, 0, dc->stream>>>(prog, fgrid, mask, off, n, cnt); break;
        case 3: qo_mc_board_kernel<3><<<grid, QO_B_TPB, 0, dc->stream>>>(prog, fgrid, mask, off, n, cnt); break;
        default: qo_mc_board_kernel<4><<<grid, QO_B_TPB, 0, dc->stream>>>(prog, fgrid, mask, off, n, cnt); break;
        }
        CU(cudaGetLastError());
        return QO_OK;
    }
    int sb, f_chunk = p->nf, n_fchunks = 1;
    if (full_s) {
        /* no per-sample reduction: cut (sample, frequency) space into ~QO_G_TPB-item tiles */
        if (p->nf >= QO_G_TPB) { sb = 1; f_chunk = QO_G_TPB; n_fchunks = (p->nf + f_chunk - 1) / f_chunk; }
        else sb = (QO_G_TPB + p->nf - 1) / p->nf;
    } else {
        sb = (2 * QO_G_TPB + p->nf - 1) / p->nf;
        if (sb < 1) sb = 1;
        /* a tile is sb * nf items dealt round-robin to QO_G_TPB threads, then a block barrier: make it a whole number of
         * rounds (nf = 3: 86 samples = 258 items left one warp working a third round for 2 items while the other three
         * waited at the barrier -- 22 % of all stall samples in profiles/r01g_generic_cfg3_details.txt; 128 samples = 3 rounds) */
        int g = QO_G_TPB, r = p->nf;
        while (r) { const int t = g % r; g = r; r = t; }
        const int step = QO_G_TPB / g;
        const int sbr = (sb + step - 1) / step * step;
        if (sbr <= QO_G_SB) sb = sbr;
    }
    if (sb > QO_G_SB) sb = QO_G_SB;
    unsigned long long tiles = ((n + sb - 1) / sb) * (unsigned long long)n_fchunks;
    unsigned long long cap = (unsigned long long)dc->sm_count * 8;
    int grid = (int)(tiles < cap ? tiles : cap);
    if (grid < 1) grid = 1;
    qo_mc_generic_kernel<<<grid, QO_G_TPB, 0, dc->stream>>>(prog, fgrid, mask, p->nf, f_chunk, n_fchunks, sb, off, n, cnt, pl, full_s);
    CU(cudaGetLastError());
    return QO_OK;
}

static int plan_launch_dev(qo_plan *p, int g, unsigned long long off, unsigned long long n, unsigned long long *cnt, qo_c64 *full_s_dev,
                           unsigned long long plane_samples, unsigned long long plane_first)
{
    if (n == 0) return QO_OK;
    CU(cudaSetDevice(p->ctx->d[g].device));
    int full_s = p->mode == QO_MODE_FULL_S;
    QoPlanes pl = { NULL, NULL, NULL, NULL, p->dev<double2>(g, p->tab.sblk), p->dev<double2>(g, p->tab.sdet), 2 * p->npairs, NULL };
    double *cplms = NULL;
    if (p->hp.cplms_elem >= 0) {
        DevCtx *dc = &p->ctx->d[g];
        CU(cudaMallocAsync((void **)&cplms, (size_t)n * 4 * sizeof(double), dc->stream));
        qo_cplms_kernel<<<(unsigned)((n + 127) / 128), 128, 0, dc->stream>>>(p->dev<DevProg>(g, p->tab.prog), off, n, cplms);
        { cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) { cudaFreeAsync(cplms, dc->stream); qo_set_error("qo_cplms_kernel launch -> %s", cudaGetErrorString(e_)); return QO_ERR_CUDA; } }
        pl.cplms = cplms;
        p->launches++;
    }
    if (full_s) {
        if (!full_s_dev) { if (cplms) cudaFreeAsync(cplms, p->ctx->d[g].stream); qo_set_error("FULL_S needs an output buffer"); return QO_ERR_ARG; }
        size_t plane = (size_t)plane_samples * (size_t)p->nf;
        double2 *base = (double2 *)full_s_dev + (size_t)plane_first * (size_t)p->nf;
        pl.s11 = base; pl.s21 = base + plane; pl.s12 = base + 2 * plane; pl.s22 = base + 3 * plane;
    }
    int rc;
    if (full_s && !p->generic && p->precision == 64 && n >= QO_FS_TF_MIN_SAMPLES && p->fs_state == 0)
        p->fs_state = qo_tf_fs_plan_check(&p->hp, 1, p->precision, p->generic, p->f.data(), p->nf, &p->ov, &p->fsp) ? 1 : -1;
    if (full_s && p->fs_state == 1 && n >= QO_FS_TF_MIN_SAMPLES) { rc = launch_tf_fs(p, g, off, n, pl); if (rc == QO_OK) p->kernel_name = "qo_fs_tf_kernel"; }
    else switch (p->kern) {
    case K_BOARD: case K_GENERIC: rc = launch_generic(p, g, off, n, cnt, pl, full_s); break;
    case K_SPOT: rc = launch_spot(p, g, off, n, cnt); break;
    case K_TF: rc = launch_tf(p, g, off, n, cnt, cplms); break;
    case K_LADDER: rc = launch_ladder(p, g, off, n, cnt, cplms); break;
    default: rc = p->precision == 32 ? launch_lumped<float>(p, g, off, n, cnt, pl, full_s) : launch_lumped<double>(p, g, off, n, cnt, pl, full_s); break;
    }
    if (cplms) cudaFreeAsync(cplms, p->ctx->d[g].stream);
    if (rc == QO_OK) p->launches++;
    return rc;
}

extern "C" int qo_plan_launch(qo_plan *p, uint64_t sample_offset, uint64_t n_samples, uint64_t *counters_dev, qo_c64 *full_s_dev)
{
    qo_clear_error();
    if (!p) return QO_ERR_ARG;
    qo_ctx *c = p->ctx;
    if (c->ndev == 1) {
        unsigned long long *cnt = counters_dev ? (unsigned long long *)counters_dev : p->counters(0);
        return plan_launch_dev(p, 0, sample_offset, n_samples, cnt, full_s_dev, n_samples, 0);
    }
    if (counters_dev || full_s_dev) { qo_set_error("caller-owned device buffers need a single-device ctx"); return QO_ERR_ARG; }
    /* shard the contiguous global sample range; Philox counters carry the GLOBAL index */
    for (int g = 0; g < c->ndev; g++) {
        unsigned long long a = n_samples * (unsigned long long)g / c->ndev, b = n_samples * (unsigned long long)(g + 1) / c->ndev;
        int rc = plan_launch_dev(p, g, sample_offset + a, b - a, p->counters(g), NULL, 0, 0);
        if (rc) return rc;
    }
    return QO_OK;
}

extern "C" int qo_plan_read(qo_plan *p, qo_mc_result *res)
{
    qo_clear_error();
    if (!p || !res) return QO_ERR_ARG;
    qo_ctx *c = p->ctx;
    std::vector<unsigned long long> h((size_t)p->ncnt, 0), tmp((size_t)p->ncnt);
    if (c->ndev > 1 && c->have_nccl) {
        /* the path's only collective: sum of u64 counters (integers => result independent of GPU count) */
        c->nccl.GroupStart();
        for (int g = 0; g < c->ndev; g++) {
            cudaSetDevice(c->d[g].device);
            int r = c->nccl.AllReduce(p->counters(g), p->counters(g), (size_t)p->ncnt, QO_NCCL_UINT64, QO_NCCL_SUM, c->comm[g], c->d[g].stream);
            if (r) { c->nccl.GroupEnd(); qo_set_error("ncclAllReduce failed (%d)", r); return QO_ERR_NCCL; }
        }
        if (c->nccl.GroupEnd()) { qo_set_error("ncclGroupEnd failed"); return QO_ERR_NCCL; }
        for (int g = 0; g < c->ndev; g++) { CU(cudaSetDevice(c->d[g].device)); CU(cudaStreamSynchronize(c->d[g].stream)); }
        CU(cudaSetDevice(c->d[0].device));
        CU(cudaMemcpy(h.data(), p->counters(0), (size_t)p->ncnt * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        /* counters now hold the global sum on every device: keep only device 0's copy as the accumulator */
        for (int g = 1; g < c->ndev; g++) { CU(cudaSetDevice(c->d[g].device)); CU(cudaMemset(p->counters(g), 0, (size_t)p->ncnt * sizeof(unsigned long long))); }
    } else {
        for (int g = 0; g < c->ndev; g++) {
            CU(cudaSetDevice(c->d[g].device));
            CU(cudaStreamSynchronize(c->d[g].stream));
            CU(cudaMemcpy(tmp.data(), p->counters(g), (size_t)p->ncnt * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            for (int i = 0; i < p->ncnt; i++) h[i] += tmp[i];
        }
    }
    res->n_pass = h[0];
    res->n_total = h[1];
    if (res->fail_per_spec) for (int s = 0; s < p->hp.nspec; s++) res->fail_per_spec[s] = h[2 + s];
    if (res->hist) for (int b = 0; b < p->hp.hist_bins; b++) res->hist[b] = h[2 + p->hp.nspec + b];
    res->flops_per_eval = p->flops_per_eval;
    return QO_OK;
}

/* ---- one-shot host-buffer entry points ------------------------------------ */
extern "C" int qo_mc_run(qo_ctx *ctx, const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec,
                         const qo_mc_cfg *cfg, qo_mc_result *res, qo_c64 *full_s)
{
    qo_clear_error();
    if (!ctx || !cfg || !res) return QO_ERR_ARG;
    if (cfg->mode == QO_MODE_FULL_S && !full_s) { qo_set_error("FULL_S needs an output buffer"); return QO_ERR_ARG; }
    if (!net || !f || nf <= 0 || (nspec > 0 && !spec) || nspec < 0) { qo_set_error("bad arguments"); return QO_ERR_ARG; }
    QoOverrides ov;
    int rc = qo_overrides_read(&ov);
    if (rc) return rc;
    /* same job and overrides as the previous call on this ctx (everything but the sample range)?  Then its plan is still good. */
    unsigned long long key = 1469598103934665603ull;
    {
        /* eight bytes per step (the grid alone is 32 KB: byte-wise FNV cost 45 us per call), bytes for the tail */
        auto mix = [&key](const void *ptr, size_t n) {
            const unsigned char *b = (const unsigned char *)ptr;
            size_t i = 0;
            for (; i + 8 <= n; i += 8) { unsigned long long w; memcpy(&w, b + i, 8); key = (key ^ w) * 0x9E3779B97F4A7C15ull; key ^= key >> 29; }
            for (; i < n; i++) { key ^= b[i]; key *= 1099511628211ull; }
        };
        mix(net->e, (size_t)net->n * sizeof(qo_elem)); mix(&net->rs, sizeof net->rs); mix(&net->rl, sizeof net->rl);
        mix(f, (size_t)nf * sizeof(double));
        if (nspec > 0) mix(spec, (size_t)nspec * sizeof(qo_spec));
        if (cfg->n_tol > 0 && cfg->tol) mix(cfg->tol, (size_t)cfg->n_tol * sizeof(qo_tol));
        const long long scal[8] = { (long long)cfg->seed, cfg->dist, cfg->n_tol, cfg->mode, cfg->precision, cfg->hist_bins, cfg->hist_spec, nspec };
        mix(scal, sizeof scal); mix(&cfg->hist_lo, sizeof(double)); mix(&cfg->hist_hi, sizeof(double));
        mix(&ov, sizeof ov);
    }
    qo_plan *p = NULL;
    static const bool mc_timing = getenv("QO100NET_MC_TIMING") != NULL;
    const auto tt0 = std::chrono::steady_clock::now();
    const bool cacheable = net->nblk == 0 && !getenv("QO100NET_NO_PLAN_CACHE");      /* measured blocks are not hashed: no reuse */
    if (cacheable && ctx->mc_cache && ctx->mc_cache_key == key && ctx->mc_cache->nf == nf) {
        p = ctx->mc_cache;
        /* the call's inputs travel host -> device every time.  Copies from pageable memory are staged by the driver (~12 us
         * each): the tables go from one page-locked copy, and the re-sends are then truly asynchronous */
        const size_t nb = p->lay.buf.size();
        if (!p->pinned) {
            if (cudaHostAlloc((void **)&p->pinned, nb, cudaHostAllocDefault) == cudaSuccess) memcpy(p->pinned, p->lay.buf.data(), nb);
            else { cudaGetLastError(); p->pinned = NULL; }
        }
        for (int g = 0; g < ctx->ndev; g++) {
            CU(cudaSetDevice(ctx->d[g].device));
            CU(cudaMemcpyAsync(p->d[g].mem, p->pinned ? (const void *)p->pinned : (const void *)p->lay.buf.data(), nb, cudaMemcpyHostToDevice, ctx->d[g].stream));
        }
        rc = qo_plan_reset(p);
        if (rc) return rc;
    } else {
        if (ctx->mc_cache) { qo_plan_destroy(ctx->mc_cache); ctx->mc_cache = NULL; }
        rc = plan_create(ctx, net, f, nf, spec, nspec, cfg, &ov, &p);
        if (rc) return rc;
        if (cacheable) { ctx->mc_cache = p; ctx->mc_cache_key = key; }
    }
    const auto tt1 = std::chrono::steady_clock::now();
    const int fs = cfg->mode == QO_MODE_FULL_S;
    const unsigned long long N = cfg->n_samples;
    qo_c64 *dbuf[8] = { 0 };
    unsigned long long a[9];
    for (int g = 0; g <= ctx->ndev; g++) a[g] = N * (unsigned long long)g / ctx->ndev;
    for (int g = 0; g < ctx->ndev && rc == QO_OK; g++) {
        cudaSetDevice(ctx->d[g].device);
        cudaEventRecord(ctx->d[g].ev0, ctx->d[g].stream);
        unsigned long long n = a[g + 1] - a[g];
        if (fs && n) {
            if (cudaMalloc(&dbuf[g], 4 * (size_t)n * nf * sizeof(qo_c64)) != cudaSuccess) { cudaGetLastError(); qo_set_error("cannot allocate %zu bytes for FULL_S output", 4 * (size_t)n * nf * sizeof(qo_c64)); rc = QO_ERR_NOMEM; break; }
        }
        rc = plan_launch_dev(p, g, cfg->sample_offset + a[g], n, p->counters(g), dbuf[g], n, 0);
        cudaEventRecord(ctx->d[g].ev1, ctx->d[g].stream);
    }
    const auto tt2 = std::chrono::steady_clock::now();
    if (rc == QO_OK) rc = qo_plan_read(p, res);
    if (mc_timing) {
        const auto tt3 = std::chrono::steady_clock::now();
        fprintf(stderr, "qo_mc_run: plan/tables %.1f us, launch %.1f us, wait+read %.1f us\n", std::chrono::duration<double, std::micro>(tt1 - tt0).count(),
                std::chrono::duration<double, std::micro>(tt2 - tt1).count(), std::chrono::duration<double, std::micro>(tt3 - tt2).count());
    }
    if (rc == QO_OK) {
        float worst = 0;
        for (int g = 0; g < ctx->ndev; g++) {
            float ms = 0;
            cudaSetDevice(ctx->d[g].device);
            cudaEventSynchronize(ctx->d[g].ev1);
            cudaEventElapsedTime(&ms, ctx->d[g].ev0, ctx->d[g].ev1);
            if (ms > worst) worst = ms;
        }
        res->seconds = worst * 1e-3;
        res->evals_per_s = res->seconds > 0 ? (double)N * nf / res->seconds : 0.0;
        if (fs) {
            res->n_total = N;
            /* planes [4][N][nf] on the host; each device holds [4][n_g][nf] */
            for (int g = 0; g < ctx->ndev && rc == QO_OK; g++) {
                unsigned long long n = a[g + 1] - a[g];
                if (!n) continue;
                cudaSetDevice(ctx->d[g].device);
                for (int pl = 0; pl < 4; pl++) {
                    cudaError_t e = cudaMemcpy(full_s + ((size_t)pl * N + a[g]) * nf, dbuf[g] + (size_t)pl * n * nf,
                                               (size_t)n * nf * sizeof(qo_c64), cudaMemcpyDeviceToHost);
                    if (e != cudaSuccess) { qo_set_error("D2H of FULL_S failed: %s", cudaGetErrorString(e)); rc = QO_ERR_CUDA; break; }
                }
            }
        }
    }
    for (int g = 0; g < ctx->ndev; g++) if (dbuf[g]) { cudaSetDevice(ctx->d[g].device); cudaFree(dbuf[g]); }
    if (rc != QO_OK || ctx->mc_cache != p) {               /* not cached, or its launch failed: do not keep it */
        if (ctx->mc_cache == p) ctx->mc_cache = NULL;
        qo_plan_destroy(p);
    }
    return rc;
}

__global__ void qo_gd_kernel(const double2 *__restrict__ s21, const double *__restrict__ f3, int nf, double *__restrict__ gd)
{
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nf) return;
    /* tau = -d(arg S21)/dw, central difference over the two bracketing points */
    double2 a = s21[nf + k], b = s21[2 * nf + k];
    double re = a.x * b.x + a.y * b.y, im = a.y * b.x - a.x * b.y;      /* a * conj(b) */
    double dw = 6.283185307179586476925286766559 * (f3[nf + k] - f3[2 * nf + k]);
    gd[k] = -atan2(im, re) / dw;
}

extern "C" int qo_sweep(qo_ctx *ctx, const qo_net *net, const double *f, int nf, int precision,
                        qo_c64 *s11, qo_c64 *s21, qo_c64 *s12, qo_c64 *s22, double *gd)
{
    qo_clear_error();
    if (!ctx || !net || !f || nf <= 0) return QO_ERR_ARG;
    if (precision != 64 && precision != 32) { qo_set_error("precision must be 64 or 32"); return QO_ERR_ARG; }
    /* group delay: evaluate f, f(1+1e-6), f(1-1e-6) in the same launch */
    const int nft = gd ? 3 * nf : nf;
    std::vector<double> f3;
    const double *fg = f;
    if (gd) {
        f3.resize((size_t)nft);
        for (int k = 0; k < nf; k++) { double df = f[k] * 1e-6; f3[k] = f[k]; f3[nf + k] = f[k] + df; f3[2 * nf + k] = f[k] - df; }
        fg = f3.data();
    }
    qo_mc_cfg cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.n_samples = 1; cfg.mode = QO_MODE_FULL_S; cfg.precision = precision;
    /* device 0 of the ctx only: a nominal sweep has nothing to shard */
    qo_ctx one = *ctx;
    one.ndev = 1;
    qo_plan *p = NULL;
    int rc = qo_plan_create(&one, net, fg, nft, NULL, 0, &cfg, &p);
    if (rc) return rc;
    DevCtx *dc = &ctx->d[0];
    double2 *buf = NULL;
    double *dgd = NULL, *df3 = NULL;
    cudaSetDevice(dc->device);
    do {
        if (cudaMallocAsync((void **)&buf, 4 * (size_t)nft * sizeof(double2), dc->stream) != cudaSuccess) { rc = QO_ERR_NOMEM; break; }
        rc = plan_launch_dev(p, 0, 0, 1, p->counters(0), (qo_c64 *)buf, 1, 0);
        if (rc) break;
        if (gd) {
            if (cudaMallocAsync((void **)&dgd, (size_t)nf * sizeof(double), dc->stream) != cudaSuccess ||
                cudaMallocAsync((void **)&df3, (size_t)nft * sizeof(double), dc->stream) != cudaSuccess) { rc = QO_ERR_NOMEM; break; }
            cudaMemcpyAsync(df3, fg, (size_t)nft * sizeof(double), cudaMemcpyHostToDevice, dc->stream);
            qo_gd_kernel<<<(nf + 127) / 128, 128, 0, dc->stream>>>(buf + (size_t)nft, df3, nf, dgd);
            p->launches++;
        }
        cudaError_t e = cudaStreamSynchronize(dc->stream);
        if (e != cudaSuccess) { qo_set_error("sweep kernel failed: %s", cudaGetErrorString(e)); rc = QO_ERR_CUDA; break; }
        qo_c64 *outs[4] = { s11, s21, s12, s22 };
        if (nft == nf && (size_t)nf * 4 * sizeof(double2) <= (1u << 20)) {
            /* one device -> host copy for all four planes (each cudaMemcpy to pageable memory costs ~10 us of latency,
             * which is what a 1024-point nominal sweep is made of), then scatter on the host */
            std::vector<double2> stage(4 * (size_t)nf);
            cudaMemcpy(stage.data(), buf, 4 * (size_t)nf * sizeof(double2), cudaMemcpyDeviceToHost);
            for (int pl = 0; pl < 4; pl++)
                if (outs[pl]) memcpy(outs[pl], stage.data() + (size_t)pl * nf, (size_t)nf * sizeof(double2));
        } else {
            for (int pl = 0; pl < 4; pl++)
                if (outs[pl]) cudaMemcpy(outs[pl], buf + (size_t)pl * nft, (size_t)nf * sizeof(double2), cudaMemcpyDeviceToHost);
        }
        if (gd) cudaMemcpy(gd, dgd, (size_t)nf * sizeof(double), cudaMemcpyDeviceToHost);
        e = cudaGetLastError();
        if (e != cudaSuccess) { qo_set_error("sweep copy failed: %s", cudaGetErrorString(e)); rc = QO_ERR_CUDA; }
    } while (0);
    if (buf) cudaFreeAsync(buf, dc->stream);
    if (dgd) cudaFreeAsync(dgd, dc->stream);
    if (df3) cudaFreeAsync(df3, dc->stream);
    qo_plan_destroy(p);
    return rc;
}

/* ---- the device's perturbation stream, for the bit-exactness test --------- */
__global__ void qo_factor_kernel(unsigned long long seed, unsigned long long off, unsigned long long n, int nvar, int dist, double tol, double *out)
{
    unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * (unsigned long long)nvar) return;
    unsigned long long s = i / (unsigned long long)nvar;
    uint32_t v = (uint32_t)(i - s * (unsigned long long)nvar);
    out[i] = QO_FMA(tol, qo_stream_variate(seed, off + s, v, dist), 1.0);
}

extern "C" int qo_device_perturb_factors(qo_ctx *ctx, uint64_t seed, uint64_t sample_offset, uint64_t n_samples,
                                         int n_var, int dist, double tol, double *out)
{
    qo_clear_error();
    if (!ctx || !out || n_var <= 0 || n_samples == 0) return QO_ERR_ARG;
    DevCtx *dc = &ctx->d[0];
    CU(cudaSetDevice(dc->device));
    size_t n = (size_t)n_samples * (size_t)n_var;
    double *d = NULL;
    CU(cudaMalloc(&d, n * sizeof(double)));
    qo_factor_kernel<<<(unsigned)((n + 255) / 256), 256, 0, dc->stream>>>(seed, sample_offset, n_samples, n_var, dist, tol, d);
    cudaError_t e = cudaStreamSynchronize(dc->stream);
    if (e == cudaSuccess) e = cudaMemcpy(out, d, n * sizeof(double), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) { qo_set_error("factor kernel: %s", cudaGetErrorString(e)); return QO_ERR_CUDA; }
    return QO_OK;
}

/* ---- the kernel's reciprocal, exposed so that its accuracy can be tested ---- */
__global__ void qo_rcp_kernel(const double *in, double *out, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = qrcp(in[i]);
}
extern "C" int qo_device_rcp(qo_ctx *ctx, const double *in, size_t n, double *out)
{
    qo_clear_error();
    if (!ctx || !in || !out || !n) return QO_ERR_ARG;
    DevCtx *dc = &ctx->d[0];
    CU(cudaSetDevice(dc->device));
    double *di = NULL, *dout = NULL;
    CU(cudaMalloc(&di, n * sizeof(double)));
    CU(cudaMalloc(&dout, n * sizeof(double)));
    cudaMemcpyAsync(di, in, n * sizeof(double), cudaMemcpyHostToDevice, dc->stream);
    qo_rcp_kernel<<<(unsigned)((n + 255) / 256), 256, 0, dc->stream>>>(di, dout, n);
    cudaError_t e = cudaStreamSynchronize(dc->stream);
    if (e == cudaSuccess) e = cudaMemcpy(out, dout, n * sizeof(double), cudaMemcpyDeviceToHost);
    cudaFree(di); cudaFree(dout);
    if (e != cudaSuccess) { qo_set_error("rcp kernel: %s", cudaGetErrorString(e)); return QO_ERR_CUDA; }
    return QO_OK;
}

__global__ void qo_mslog_kernel(const double *in, double *out, size_t n)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = ms_log(in[i]);
}
extern "C" int qo_device_mslog(qo_ctx *ctx, const double *in, size_t n, double *out)
{
    qo_clear_error();
    if (!ctx || !in || !out || !n) return QO_ERR_ARG;
    DevCtx *dc = &ctx->d[0];
    CU(cudaSetDevice(dc->device));
    double *di = NULL, *dout = NULL;
    CU(cudaMalloc(&di, n * sizeof(double)));
    CU(cudaMalloc(&dout, n * sizeof(double)));
    cudaMemcpyAsync(di, in, n * sizeof(double), cudaMemcpyHostToDevice, dc->stream);
    qo_mslog_kernel<<<(unsigned)((n + 255) / 256), 256, 0, dc->stream>>>(di, dout, n);
    cudaError_t e = cudaStreamSynchronize(dc->stream);
    if (e == cudaSuccess) e = cudaMemcpy(out, dout, n * sizeof(double), cudaMemcpyDeviceToHost);
    cudaFree(di); cudaFree(dout);
    if (e != cudaSuccess) { qo_set_error("log kernel: %s", cudaGetErrorString(e)); return QO_ERR_CUDA; }
    return QO_OK;
}

/* ---- FP64 FMA peak: dependency-free DFMA loop (roofline denominator) ------- */
__global__ void __launch_bounds__(256) qo_dfma_peak_kernel(double *out, int iters, double x, double y)
{
    double a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            a0 = fma(a0, x, y); a1 = fma(a1, x, y); a2 = fma(a2, x, y); a3 = fma(a3, x, y);
            a4 = fma(a4, x, y); a5 = fma(a5, x, y); a6 = fma(a6, x, y); a7 = fma(a7, x, y);
        }
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

extern "C" int qo_measure_dfma_peak(qo_ctx *ctx, double *tflops)
{
    qo_clear_error();
    if (!ctx || !tflops) return QO_ERR_ARG;
    DevCtx *dc = &ctx->d[0];
    CU(cudaSetDevice(dc->device));
    const int blocks = dc->sm_count * 8, iters = 4096;
    double *d = NULL;
    CU(cudaMalloc(&d, (size_t)blocks * 256 * sizeof(double)));
    double best = 0;
    for (int rep = 0; rep < 6; rep++) {
        cudaEventRecord(dc->ev0, dc->stream);
        qo_dfma_peak_kernel<<<blocks, 256, 0, dc->stream>>>(d, iters, 0.999999, 1e-9);
        cudaEventRecord(dc->ev1, dc->stream);
        cudaError_t e = cudaEventSynchronize(dc->ev1);
        if (e != cudaSuccess) { cudaFree(d); qo_set_error("dfma kernel: %s", cudaGetErrorString(e)); return QO_ERR_CUDA; }
        float ms = 0;
        cudaEventElapsedTime(&ms, dc->ev0, dc->ev1);
        double tf = (double)blocks * 256 * iters * 64 * 2 / (ms * 1e-3) * 1e-12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaFree(d);
    *tflops = best;
    return QO_OK;
}
