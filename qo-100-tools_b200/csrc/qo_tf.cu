/*
 * qo_tf.cu -- instantiations, launcher and plan-time self-check of the transfer-function kernel (qo_tf.cuh).
 * Its own translation unit (compiles in parallel with qo_cuda.cu / qo_ladder.cu).
 */
#include <cuda_runtime.h>
#include <complex>
#include <vector>
#include <mutex>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "qo_tf.cuh"
#include "qo_spot.cuh"
#include "qo_tf_fs.cuh"
#include "qo_tf_launch.h"
#include "qo_overrides.h"

/* launch shapes (profiles/r01h_*): plain ladders run 8 points per thread (coefficient loads and loop
 * overhead amortised over 8 Horner sets), the four-chain modes (coupler block, |S11| specs) 4 */
#define QO_TF_PP 4
#define QO_TF_TPB 128
#define QO_TF_MINB 4
#define QO_TF_CPL_PP 2
#define QO_TF_CPL_TPB 128
#define QO_TF_CPL_MINB 4

typedef void (*tf_fn)(const TfParams);
/* qo_tf_front.cu: a line / measured two-port in front, and |S11| specs behind any front block (their own translation unit: build time) */
tf_fn qo_tf_pick_front(int front, int s11, int pp, int den, int nspec, int *tpb, int *minb);

/* pairs per thread per iteration: short grids take one pair per thread (iterations of 64 points) so that the padding to whole
 * iterations does not dominate -- 8 points per thread are ~25 % cheaper per point but pad to 512 */
extern "C" int qo_tf_default_pp(const TfPlan *tp, int npairs)
{
    if (tp->nn == 4) return npairs <= 32 ? 1 : QO_TF_CPL_PP;
    return npairs <= 192 ? 1 : QO_TF_PP;
}

template <int NN, int CPL, bool S11, int NS, int PP, int TPB, int MINB> static tf_fn tf_pick_ns(int den)
{
    switch (den) {
    case QO_TF_DEN_NONE: return qo_mc_tf_kernel<NN, QO_TF_DEN_NONE, CPL, S11, false, NS, PP, TPB, MINB>;
    case QO_TF_DEN_E: return qo_mc_tf_kernel<NN, QO_TF_DEN_E, CPL, S11, false, NS, PP, TPB, MINB>;
    case QO_TF_DEN_D: return qo_mc_tf_kernel<NN, QO_TF_DEN_D, CPL, S11, false, NS, PP, TPB, MINB>;
    default: return nullptr;
    }
}
template <int NN, int CPL, bool S11, int PP, int TPB, int MINB> static tf_fn tf_pick(int den, int nspec = 4)
{
    return nspec > 4 ? tf_pick_ns<NN, CPL, S11, 8, PP, TPB, MINB>(den) : tf_pick_ns<NN, CPL, S11, 4, PP, TPB, MINB>(den);
}
template <int NS, int PP, int TPB, int MINB> static tf_fn tf_pick_gd_ns(int den)
{
    switch (den) {
    case QO_TF_DEN_NONE: return qo_mc_tf_kernel<4, QO_TF_DEN_NONE, 0, false, true, NS, PP, TPB, MINB>;
    case QO_TF_DEN_DD: return qo_mc_tf_kernel<4, QO_TF_DEN_DD, 0, false, true, NS, PP, TPB, MINB>;
    default: return nullptr;
    }
}
template <int PP, int TPB, int MINB> static tf_fn tf_pick_gd(int den, int nspec)
{
    return nspec > 4 ? tf_pick_gd_ns<8, PP, TPB, MINB>(den) : tf_pick_gd_ns<4, PP, TPB, MINB>(den);
}

extern "C" int qo_tf_launch(const TfPlan *tp, int pp, int sm_count, const TfParams *P, cudaStream_t st)
{
    tf_fn fn = nullptr;
    int tpb = QO_TF_TPB, minb = QO_TF_MINB;
    const bool rot = P->cpl_lin && P->cpl_matched;      /* coupler on a uniformly spaced grid: angles by rotation */
    /* a line / measured block in front, or |S11| specs behind any front block: qo_tf_front.cu (checked FIRST: the plain
     * |S11| instantiations below know nothing about a block) */
    if (tp->nn == 4 && tp->cpl_op >= 0 && (tp->front || tp->s11)) fn = qo_tf_pick_front(tp->front, tp->s11, pp, tp->den, P->nspec, &tpb, &minb);
    else if (tp->nn == 2 && pp == QO_TF_PP) fn = tf_pick<2, 0, false, QO_TF_PP, QO_TF_TPB, QO_TF_MINB>(tp->den, P->nspec);
    else if (tp->nn == 2 && pp == 1) fn = tf_pick<2, 0, false, 1, QO_TF_TPB, QO_TF_MINB>(tp->den, P->nspec);
    else if (tp->gd && pp == 1) fn = tf_pick_gd<1, QO_TF_TPB, QO_TF_MINB>(tp->den, P->nspec);
    else if (tp->nn == 4 && tp->s11 && pp == 1) fn = tf_pick<4, 0, true, 1, QO_TF_TPB, QO_TF_MINB>(tp->den, P->nspec);
    else if (tp->nn == 4 && !tp->s11 && pp == 1) fn = rot ? (P->cpl_same ? tf_pick<4, 3, false, 1, QO_TF_TPB, QO_TF_MINB>(tp->den, P->nspec) : tf_pick<4, 2, false, 1, QO_TF_TPB, QO_TF_MINB>(tp->den, P->nspec))
                 : tf_pick<4, 1, false, 1, QO_TF_TPB, QO_TF_MINB>(tp->den, P->nspec);
    else if (tp->gd && pp == QO_TF_CPL_PP) { fn = tf_pick_gd<QO_TF_CPL_PP, QO_TF_CPL_TPB, QO_TF_CPL_MINB>(tp->den, P->nspec); tpb = QO_TF_CPL_TPB; minb = QO_TF_CPL_MINB; }
    else if (tp->nn == 4 && tp->s11 && pp == QO_TF_CPL_PP) { fn = tf_pick<4, 0, true, QO_TF_CPL_PP, QO_TF_CPL_TPB, QO_TF_CPL_MINB>(tp->den, P->nspec); tpb = QO_TF_CPL_TPB; minb = QO_TF_CPL_MINB; }
    else if (tp->nn == 4 && !tp->s11 && pp == QO_TF_CPL_PP) {
        fn = rot ? (P->cpl_same ? tf_pick<4, 3, false, QO_TF_CPL_PP, QO_TF_CPL_TPB, QO_TF_CPL_MINB>(tp->den, P->nspec)
                                : tf_pick<4, 2, false, QO_TF_CPL_PP, QO_TF_CPL_TPB, QO_TF_CPL_MINB>(tp->den, P->nspec))
                 : tf_pick<4, 1, false, QO_TF_CPL_PP, QO_TF_CPL_TPB, QO_TF_CPL_MINB>(tp->den, P->nspec);
        tpb = QO_TF_CPL_TPB; minb = QO_TF_CPL_MINB;
    }
    if (!fn) return -1;
    const unsigned long long warps = (unsigned long long)(tpb / 32);
    unsigned long long blocks = (P->nsamples + warps - 1) / warps;
    const unsigned long long resident = (unsigned long long)sm_count * (unsigned long long)minb;
    if (blocks > resident) blocks = resident;
    if (blocks < 1) blocks = 1;
    fn<<<(unsigned)blocks, tpb, 0, st>>>(*P);
    return (int)cudaGetLastError();
}

extern "C" int qo_spot_launch(int need_s11, int sm_count, const SpotParams *P, cudaStream_t st)
{
    unsigned long long blocks = (P->nsamples + QO_SPOT_TPB - 1) / QO_SPOT_TPB;
    const unsigned long long cap = (unsigned long long)sm_count * 4 * 8;        /* 8 waves of resident blocks, grid-stride beyond */
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    if (need_s11) qo_mc_spot_kernel<true><<<(unsigned)blocks, QO_SPOT_TPB, 0, st>>>(*P);
    else qo_mc_spot_kernel<false><<<(unsigned)blocks, QO_SPOT_TPB, 0, st>>>(*P);
    return (int)cudaGetLastError();
}

/* ---- plan-time self-check (host) ------------------------------------------------------------------------- */
typedef std::complex<double> cplx;

/* the device's expansion, in the same order and with the same normalisation */
static void tf_expand_host(const double (*rec)[QO_TF_REC], int n_el, double rl, double zn, double *p, double *q, double *d, double *ee)
{
    const int NC = 2 * QO_TF_MAXK + 2;
    for (int i = 0; i < NC; i++) p[i] = q[i] = d[i] = 0.0;
    p[0] = rl; q[0] = zn; d[0] = 1.0;
    /* E(y) = prod_e (E0 + E1 y + E2 y^2), all 2 n_el + 1 coefficients (the kernel keeps the first K) */
    const int NE = 2 * QO_TF_MAXEL + 1;
    for (int i = 0; i < NE; i++) ee[i] = 0.0;
    ee[0] = 1.0;
    for (int e = n_el - 1; e >= 0; e--) {
        double ne[2 * QO_TF_MAXEL + 1];
        for (int i = 0; i < NE; i++)
            ne[i] = fma(rec[e][6], ee[i], fma(rec[e][7], i >= 1 ? ee[i - 1] : 0.0, rec[e][8] * (i >= 2 ? ee[i - 2] : 0.0)));
        for (int i = 0; i < NE; i++) ee[i] = ne[i];
    }
    std::vector<double> na(NC), nb(NC), ndv(NC);
    for (int e = n_el - 1; e >= 0; e--) {
        const double *r = rec[e];
        const bool series = r[9] != 0.0;
        double *a = series ? p : q, *b = series ? q : p;
        for (int i = 0; i < NC; i++) {
            const double a1 = i >= 1 ? a[i - 1] : 0.0, a2 = i >= 2 ? a[i - 2] : 0.0, b1 = i >= 1 ? b[i - 1] : 0.0, b2 = i >= 2 ? b[i - 2] : 0.0;
            const double d1 = i >= 1 ? d[i - 1] : 0.0, d2 = i >= 2 ? d[i - 2] : 0.0;
            double v = fma(r[3], a[i], fma(r[4], a1, r[5] * a2));
            na[i] = fma(r[0], b[i], fma(r[1], b1, fma(r[2], b2, v)));
            nb[i] = fma(r[3], b[i], fma(r[4], b1, r[5] * b2));
            ndv[i] = fma(r[3], d[i], fma(r[4], d1, r[5] * d2));
        }
        for (int i = 0; i < NC; i++) { a[i] = na[i]; b[i] = nb[i]; d[i] = ndv[i]; }
    }
}

static cplx tf_horner_host(const double *c, int K, double x)
{
    const double y = -x * x;
    double re = c[2 * (K - 1)], im = c[2 * (K - 1) + 1];
    /* plain multiply-add: this is a conditioning check, not a bit-exact twin, and fma() is a libm call on the host */
    for (int k = K - 2; k >= 0; k--) { re = re * y + c[2 * k]; im = im * y + c[2 * k + 1]; }
    return cplx(re, im * x);
}

/* |poly(jx)| bookkeeping of one corner of the tolerance box */
struct TfCorner {
    double rec[QO_TF_MAXEL][QO_TF_REC];
    double nd[QO_TF_MAXEL][6];
    int ser[QO_TF_MAXEL];
    double pp[2 * QO_TF_MAXK + 2], qq[2 * QO_TF_MAXK + 2], dd[2 * QO_TF_MAXK + 2], ee[2 * QO_TF_MAXEL + 1];
};

static int tf_plan_check_uncached(const DevProg *hp, int mode_reduce_only, int precision, int generic, const double *f, int nf,
                                  const unsigned char *mask, const QoOverrides *ov, TfPlan *out);

/* Fused margins (qo_tf_fuse) for the thread-per-sample kernel.  A |S21| spec other than the histogram's is fused when, at every
 * corner of the analysis and every grid point where it is the only spec that looks, the host twin of the device's F (same
 * coefficients, same formation, same Horner) stays within QO_TF_FUSE_TOL of |den|^2 of the unfused margin N2 - t E evaluated
 * from the same truncated polynomials in long double.  A stop band passes easily (~1e-13); the pass band of a ripple filter
 * usually does not, |Num|^2 cancelling inside the ripple (~1e-11). */
#define QO_TF_FUSE_TOL 1e-12
static void tf_fuse_gate(const DevProg *hp, int nf, const double *xg, const unsigned char *mask, const std::vector<TfCorner> &cs,
                         double zni, TfPlan *out)
{
    out->fused = 0; out->fused_err = 0.0;
    if (out->cpl_op >= 0 || !qo_ts_eligible(out, hp->nspec, 0)) return;
    const int kn = out->kn, ke = out->den == QO_TF_DEN_E ? out->kd : 0, nfz = 2 * kn > ke ? 2 * kn : ke;
    const double zq0 = hp->rs * zni;
    for (int s = 0; s < hp->nspec; s++) {
        if (hp->spec_kind[s] != SK_DEN2_MAX && hp->spec_kind[s] != SK_DEN2_MIN) continue;
        if (hp->hist_bins > 0 && hp->hist_spec == s) continue;
        const bool neg = hp->spec_kind[s] == SK_DEN2_MIN;
        const double t = hp->spec_thr[s];
        double worst = 0.0;
        int npts = 0;
        for (size_t ci = 0; ci < cs.size(); ci++) {
            double cn[2 * QO_TF_MAXK], fz[2 * QO_TF_MAXK + QO_TF_MAXKE];
            for (int i = 0; i < 2 * kn; i++) cn[i] = fma(zq0, cs[ci].qq[i], cs[ci].pp[i]);      /* the device's numerator pairs */
            qo_tf_fuse(kn, ke, cn, cs[ci].ee, t, neg, fz);
            for (int k = 0; k < nf; k++) {
                if (mask[k] != 1u << s) continue;
                npts++;
                const double x = xg[k], y = -(x * x);
                double got = fz[nfz - 1];
                for (int m = nfz - 2; m >= 0; m--) got = fma(got, y, fz[m]);
                const long double yl = y;
                long double r0 = cn[2 * kn - 2], r1 = cn[2 * kn - 1], e = ke > 0 ? cs[ci].ee[ke - 1] : 1.0;
                for (int i = kn - 2; i >= 0; i--) { r0 = r0 * yl + cn[2 * i]; r1 = r1 * yl + cn[2 * i + 1]; }
                for (int m = ke - 2; m >= 0; m--) e = e * yl + cs[ci].ee[m];
                const long double n2 = r0 * r0 - yl * r1 * r1, ref = neg ? n2 - t * e : t * e - n2;
                double err = (double)(fabsl((long double)got - ref) / n2);
                if (!(err == err)) err = 1e300;
                if (err > worst) worst = err;
            }
        }
        if (npts > 0 && worst <= QO_TF_FUSE_TOL) {
            out->fused |= 1u << s;
            if (worst > out->fused_err) out->fused_err = worst;
        }
    }
}

/* Where in the tolerance box the analysis looks (x[v] in [-1, 1] per random variable):
 *   0 every variable at -1, 1 the nominal network, 2 every variable at +1,
 *   3 every variable at the end that RAISES the parameters it drives (lowest self-resonances: L, C up whatever the sign of
 *     the tolerance entry), 4 its mirror image,
 *   5 .. 5+QO_TF_NVERT-1  pseudo-random vertices (each variable +-1: mixed corners such as L up / C down),
 *   then QO_TF_NINT pseudo-random interior points.
 * The choice is a fixed Philox stream, so the analysis is deterministic and cacheable. */
#define QO_TF_NVERT 20
#define QO_TF_NINT 8
#define QO_TF_NCORNER (5 + QO_TF_NVERT + QO_TF_NINT)
#define QO_TF_NOMINAL 1
static void tf_corner_vars(const DevProg *hp, int e0, int nl, int ci, double *x)
{
    const unsigned long long key = 0x51ed270b7f4a7c15ull;
    for (int v = 0; v < QO_MAX_VAR; v++) {
        if (ci == 0) x[v] = -1.0;
        else if (ci == 1) x[v] = 0.0;
        else if (ci == 2) x[v] = 1.0;
        else if (ci < 5) x[v] = 0.0;                                  /* filled below */
        else if (ci < 5 + QO_TF_NVERT) x[v] = qo_stream_variate(key, (unsigned long long)ci, (uint32_t)v, 0 /* uniform */) < 0.0 ? -1.0 : 1.0;
        else x[v] = qo_stream_variate(key, (unsigned long long)ci, (uint32_t)v, 0 /* uniform */);
    }
    if (ci == 3 || ci == 4)
        for (int e = nl - 1; e >= 0; e--)
            for (int k = 5; k >= 0; k--) {                           /* p[0] (the L or C value) decides last */
                const int v = hp->tvar[e0 + e][k];
                if (v >= 0 && hp->ttol[e0 + e][k] != 0.0) x[v] = ((hp->ttol[e0 + e][k] > 0.0) == (ci == 3)) ? 1.0 : -1.0;
            }
}

/* The analysis is a pure function of (program, grid, masks, overrides); callers that run the same job
 * repeatedly through qo_mc_run (one plan per call) would redo ~2 ms of host work per call, so the last few results
 * are kept, keyed by a 64-bit FNV-1a hash of those inputs. */
static unsigned long long tf_fnv(unsigned long long h, const void *p, size_t n)
{
    const unsigned char *b = (const unsigned char *)p;
    for (size_t i = 0; i < n; i++) { h ^= b[i]; h *= 1099511628211ull; }
    return h;
}
struct TfCacheEntry { unsigned long long key; int used, sel; TfPlan plan; };
static TfCacheEntry tf_cache[8];
static int tf_cache_next;
static std::mutex tf_cache_mu;

extern "C" int qo_tf_plan_check(const DevProg *hp, int mode_reduce_only, int precision, int generic, const double *f, int nf,
                                const unsigned char *mask, const QoOverrides *ov, TfPlan *out)
{
    /* the cheap refusals first: nominal sweeps and FULL_S jobs come through here too and must not pay for the hash */
    if (generic || !mode_reduce_only || precision != 64) return tf_plan_check_uncached(hp, mode_reduce_only, precision, generic, f, nf, mask, ov, out);
    unsigned long long key = 1469598103934665603ull;
    {
        /* what the analysis does not read must not split the cache: seed, distribution, histogram range, user limits (the
         * fused-margin gate reads the canonical thresholds and which spec the histogram tracks) */
        DevProg *k = new DevProg(*hp);
        k->seed = 0; k->dist = 0; k->hist_lo = k->hist_hi = 0.0;
        if (k->hist_bins <= 0) k->hist_spec = k->hist_bins = 0;
        else k->hist_bins = 1;
        for (int s = 0; s < QO_NSPEC_MAX; s++) k->spec_limit[s] = 0.0;
        key = tf_fnv(key, k, sizeof *k);
        delete k;
    }
    key = tf_fnv(key, f, (size_t)nf * sizeof(double));
    key = tf_fnv(key, mask, (size_t)nf);
    const int scal[4] = { mode_reduce_only, precision, generic, nf };
    key = tf_fnv(key, scal, sizeof scal);
    key = tf_fnv(key, ov, sizeof *ov);
    {
        std::lock_guard<std::mutex> lk(tf_cache_mu);
        for (int i = 0; i < 8; i++)
            if (tf_cache[i].used && tf_cache[i].key == key) { *out = tf_cache[i].plan; return tf_cache[i].sel; }
    }
    const int sel = tf_plan_check_uncached(hp, mode_reduce_only, precision, generic, f, nf, mask, ov, out);
    {
        std::lock_guard<std::mutex> lk(tf_cache_mu);
        TfCacheEntry &e = tf_cache[tf_cache_next];
        tf_cache_next = (tf_cache_next + 1) & 7;
        e.key = key; e.used = 1; e.sel = sel; e.plan = *out;
    }
    return sel;
}

static int tf_plan_check_uncached(const DevProg *hp, int mode_reduce_only, int precision, int generic, const double *f, int nf,
                                  const unsigned char *mask, const QoOverrides *ov, TfPlan *out)
{
    memset(out, 0, sizeof *out);
    out->cpl_op = -1;
#define QO_TF_NO(msg) do { out->reason = msg; return 0; } while (0)
    if (ov->kernel == QoOverrides::INTERP || ov->kernel == QoOverrides::LADDER) QO_TF_NO("QO100NET_KERNEL override");
    if (generic || !mode_reduce_only || precision != 64) QO_TF_NO("not a reduce-only FP64 job on a lumped cascade");
    if (hp->nspec < 1 || hp->nspec > QO_TF_NSPEC || hp->n_var > QO_MAX_VAR) QO_TF_NO("spec / variable count");
    for (int s = 0; s < hp->nspec; s++)
        if (hp->spec_kind[s] != SK_DEN2_MAX && hp->spec_kind[s] != SK_DEN2_MIN && hp->spec_kind[s] != SK_S11_MAX && hp->spec_kind[s] != SK_GD_MAX) QO_TF_NO("spec kind");
    int need_s21 = 0;
    for (int s = 0; s < hp->nspec; s++) if (hp->spec_kind[s] != SK_S11_MAX) need_s21 = 1;      /* group delay needs D too */
    const bool gd = hp->need_gd != 0;
    int e0 = hp->op0;
    /* one non-rational block may sit in FRONT of the lumped ops (source side): a coupled-line section, a transmission line or a
     * measured two-port.  Its row vector [1 Rs] M_block is evaluated per point (closed form / per-frequency table) and
     * contracted with the polynomials [P; Q] of everything behind it */
    if (hp->n_ops > e0 && hp->opcode[e0] == OP_CPL) { out->cpl_op = e0; out->front = 0; e0++; }
    else if (hp->n_ops > e0 + 1 && hp->opcode[e0] == OP_TLINE && !ov->tf_no_front) { out->cpl_op = e0; out->front = 1; e0++; }
    else if (hp->n_ops > e0 + 1 && hp->opcode[e0] == OP_SBLOCK && !ov->tf_no_front) { out->cpl_op = e0; out->front = 2; e0++; }
    const int nl = hp->n_ops - e0;
    if (nl < 1 || nl > QO_TF_MAXEL) QO_TF_NO("element count");
    int deg = 0, has_d = 0;
    for (int e = 0; e < nl; e++) {
        const int op = hp->opcode[e0 + e], dg = qo_tf_degree(op);
        if (dg < 0) QO_TF_NO("non-lumped element");
        deg += dg;
        if (!(op == OP_SER_R || op == OP_SER_L || op == OP_SHUNT_C)) has_d = 1;     /* these have D == 1 exactly */
    }
    if (deg > 2 * QO_TF_MAXK - 1) QO_TF_NO("polynomial degree");
    const int Kfull = deg / 2 + 1;
    const bool cpl = out->cpl_op >= 0, s11 = hp->need_s11 != 0;
    if (gd && (cpl || s11)) QO_TF_NO("group-delay specs mixed with a front block or |S11| specs");
    if (!need_s21) has_d = 0;                                 /* S11 = (P - Rs Q) / (P + Rs Q): the branch denominators cancel */
    const bool apart = cpl || s11;                            /* P and Q kept apart */
    out->deg = deg; out->el0 = e0; out->n_el = nl; out->nn = (apart || gd) ? 4 : 2; out->s11 = s11; out->gd = gd;

    const double two_pi = 6.283185307179586476925286766559;
    double fmin = f[0], fmax = f[0];
    for (int k = 1; k < nf; k++) { if (f[k] < fmin) fmin = f[k]; if (f[k] > fmax) fmax = f[k]; }
    const double wr = two_pi * sqrt(fmin * fmax);
    out->wref = wr;
    const double zn = sqrt(hp->rs * hp->rl), zni = 1.0 / zn;

    /* expansions of the nominal network and of QO_TF_NCORNER - 1 other points of the tolerance box (tf_corner_vars) */
    const int NCORN = hp->n_var > 0 ? QO_TF_NCORNER : 2;          /* no tolerances: every "corner" is the nominal network */
    std::vector<TfCorner> cs((size_t)NCORN);
    for (int ci = 0; ci < NCORN; ci++) {
        TfCorner &c = cs[ci];
        double xv[QO_MAX_VAR];
        tf_corner_vars(hp, e0, nl, ci, xv);
        for (int e = 0; e < nl; e++) {
            double p[6];
            for (int k = 0; k < 6; k++) {
                p[k] = hp->nom[e0 + e][k];
                if (hp->tvar[e0 + e][k] >= 0) p[k] = qo_stream_apply(p[k], hp->ttol[e0 + e][k], xv[hp->tvar[e0 + e][k]], hp->tmode[e0 + e][k]);
            }
            c.ser[e] = qo_tf_element(hp->opcode[e0 + e], p, wr, c.nd[e]);
            const double sc = c.ser[e] ? zni : zn;
            const double *nd = c.nd[e];
            double *rec = c.rec[e];
            rec[0] = nd[0] * sc; rec[1] = nd[1] * sc; rec[2] = nd[2] * sc; rec[3] = nd[3]; rec[4] = nd[4]; rec[5] = nd[5];
            rec[6] = nd[3] * nd[3]; rec[7] = fma(2.0 * nd[3], nd[5], -nd[4] * nd[4]); rec[8] = nd[5] * nd[5];
            rec[9] = c.ser[e] ? 1.0 : 0.0;
        }
        tf_expand_host(c.rec, nl, hp->rl, zn, c.pp, c.qq, c.dd, c.ee);
        for (int i = 2 * Kfull; i < 2 * QO_TF_MAXK + 2; i++)
            if (c.pp[i] != 0.0 || c.qq[i] != 0.0 || c.dd[i] != 0.0) QO_TF_NO("degree accounting");
    }

    /* Polynomial lengths: keep the terms the grid can see.  A kept length is accepted when the terms it drops add up to
     * less than `trunc` (relative) at every grid point of all three expansions -- numerators against |P| + zn |Q|
     * (|Num| for plain ladders), D against |D|, E against E.  QO100NET_TF_TRUNC=0 keeps everything.
     * Per point the scan runs from the top coefficient down and stops at the first term that may not be dropped. */
    const double trunc = gd ? 0.0 : ov->tf_trunc;          /* the derivative polynomials weigh the top coefficients by their index: keep all */
    const int NE = 2 * nl + 1, NC = 2 * Kfull;
    int kn = 1, kdd = 1, ke = 1;
    std::vector<double> xg((size_t)nf), xpw((size_t)NC + 1), zpw((size_t)NE + 1);
    for (int k = 0; k < nf; k++) xg[k] = two_pi * f[k] / wr;
    /* |coefficient| tables of the three expansions (numerator entry: what the device's Num / [P; Q] pair carries) */
    std::vector<double> an((size_t)NCORN * NC), ad((size_t)NCORN * NC), ae((size_t)NCORN * NE);
    for (int ci = 0; ci < NCORN; ci++)
        for (int i = 0; i < NC; i++) {
            an[(size_t)ci * NC + i] = apart ? fabs(cs[ci].pp[i]) + fabs(cs[ci].qq[i]) : fabs(cs[ci].pp[i] + hp->rs * zni * cs[ci].qq[i]);
            ad[(size_t)ci * NC + i] = fabs(cs[ci].dd[i]);
        }
    for (int ci = 0; ci < NCORN; ci++)
        for (int m = 0; m < NE; m++) ae[(size_t)ci * NE + m] = fabs(cs[ci].ee[m]);
    for (int k = 0; k < nf; k++) {
        const double x = xg[k], x2 = x * x;
        xpw[0] = 1.0; for (int i = 1; i <= NC; i++) xpw[i] = xpw[i - 1] * x;
        zpw[0] = 1.0; for (int m = 1; m <= NE; m++) zpw[m] = zpw[m - 1] * x2;
        for (int ci = 0; ci < NCORN; ci++) {
            /* the three classic corners on every grid point, the others on every 4th and at the grid's ends (tails are smooth in x) */
            if (ci > 2 && (k & 3) && k + 1 < nf) continue;
            const TfCorner &c = cs[ci];
            const cplx P_ = tf_horner_host(c.pp, Kfull, x), Q_ = tf_horner_host(c.qq, Kfull, x) * zni, D_ = tf_horner_host(c.dd, Kfull, x);
            const double nref = trunc * (apart ? sqrt(std::norm(P_)) + zn * sqrt(std::norm(Q_)) : sqrt(std::norm(P_ + hp->rs * Q_)));
            const double dref = trunc * sqrt(std::norm(D_));
            const double *pn = &an[(size_t)ci * NC], *pd = &ad[(size_t)ci * NC], *pe = &ae[(size_t)ci * NE];
            /* numerators: drop whole pairs (2K, 2K+1) from the top while their sum stays below the bound */
            double acc = 0.0;
            int K = Kfull;
            while (K > kn) { acc += pn[2 * K - 1] * xpw[2 * K - 1] + pn[2 * K - 2] * xpw[2 * K - 2]; if (acc > nref) break; K--; }
            if (K > kn) kn = K;
            if (has_d) {
                acc = 0.0; K = Kfull;
                while (K > kdd) { acc += pd[2 * K - 1] * xpw[2 * K - 1] + pd[2 * K - 2] * xpw[2 * K - 2]; if (acc > dref) break; K--; }
                if (K > kdd) kdd = K;
                double full = 0.0;
                for (int m = 0; m < NE; m++) full += c.ee[m] * (m & 1 ? -zpw[m] : zpw[m]);
                const double eref = trunc * full;
                acc = 0.0; K = NE;
                while (K > ke) { acc += pe[K - 1] * zpw[K - 1]; if (!(acc <= eref)) break; K--; }
                if (K > ke) ke = K;
            }
        }
    }
    ke = (ke + 1) & ~1;                                       /* the kernel loads E two coefficients at a time */
    if (ke < 2) ke = 2;
    if (kn < 2) kn = 2;                                       /* the Horner code starts from the two top rows (a zero row costs one FMA) */
    if (kdd < 2) kdd = 2;
    out->kn = kn;
    /* denominator form: the truncated |D|^2 polynomial when it is short enough to pay, else D itself; a form whose
     * self-check fails (E loses digits next to a trap's notch, where |D| -> 0) hands over to the next one */
    int forms[2], nforms = 0;
    if (!has_d) forms[nforms++] = QO_TF_DEN_NONE;
    else if (gd) forms[nforms++] = QO_TF_DEN_DD;
    else {
        if (ke <= QO_TF_MAXKE && ke <= 2 * kdd + 3) forms[nforms++] = QO_TF_DEN_E;
        forms[nforms++] = QO_TF_DEN_D;
    }
    const double tol = ov->tf_tol;
    double worst = 0.0;
    int accepted = 0;
    for (int fi = 0; fi < nforms && !accepted; fi++) {
        out->den = forms[fi];
        out->kd = forms[fi] == QO_TF_DEN_E ? ke : (forms[fi] == QO_TF_DEN_D || forms[fi] == QO_TF_DEN_DD) ? kdd : 0;
        /* self-check: exactly what the device evaluates (kept lengths, this denominator form) against the per-element evaluation */
        worst = 0.0;
        int range_ok = 1;
        for (int ci = 0; ci < NCORN && range_ok; ci++) {
            const TfCorner &c = cs[ci];
            for (int k = 0; k < nf; k++) {
                const double x = xg[k], y = -x * x;
                if (ci > 2 && (k & 3) && k > 0 && k + 1 < nf && mask[k - 1] == mask[k] && mask[k + 1] == mask[k]) continue;
                double d2 = 1.0;
                if (out->den == QO_TF_DEN_E) { d2 = c.ee[out->kd - 1]; for (int m = out->kd - 2; m >= 0; m--) d2 = d2 * y + c.ee[m]; }
                else if (out->den == QO_TF_DEN_D || out->den == QO_TF_DEN_DD) d2 = std::norm(tf_horner_host(c.dd, out->kd, x));
                if (!(d2 > 1e-70 && d2 < 1e70)) { range_ok = 0; break; }      /* the batched reciprocal multiplies four of them */
                /* value check: every in-band point of the nominal network; every other point of the box on every 4th point and
                 * around the band edges (their job is to catch a tolerance-driven loss of conditioning, which is smooth in x) */
                if (!mask[k]) continue;
                if (ci != QO_TF_NOMINAL && (k & 3) && k > 0 && k + 1 < nf && mask[k - 1] == mask[k] && mask[k + 1] == mask[k]) continue;
                const cplx P_ = tf_horner_host(c.pp, kn, x), Q_ = tf_horner_host(c.qq, kn, x) * zni;
                /* per-element evaluation, column vector from the load end: imm = N(jx) / D(jx) */
                double ar = hp->rl, ai = 0.0, br = 1.0, bi = 0.0, dref = 1.0;
                for (int e = nl - 1; e >= 0; e--) {
                    const double *nd = c.nd[e];
                    const double nr = nd[2] * y + nd[0], ni = nd[1] * x, dr = nd[5] * y + nd[3], di = nd[4] * x;
                    const double dn = dr * dr + di * di, inv = 1.0 / dn;
                    const double ir = (nr * dr + ni * di) * inv, ii = (ni * dr - nr * di) * inv;
                    if (c.ser[e]) { const double tr = ir * br - ii * bi, ti = ir * bi + ii * br; ar += tr; ai += ti; }
                    else { const double tr = ir * ar - ii * ai, ti = ir * ai + ii * ar; br += tr; bi += ti; }
                    dref *= dn;
                }
                const cplx a(ar, ai), b(br, bi);
                double rel;
                if (cpl) {
                    /* P/D and Q/D as complex numbers (the coupler's row vector mixes them), plus the kernel's |D|^2 against the true one */
                    const cplx Dc = tf_horner_host(c.dd, Kfull, x);
                    rel = 2.0 * (std::abs(P_ / Dc - a) + zn * std::abs(Q_ / Dc - b)) / (std::abs(a) + zn * std::abs(b)) + (need_s21 ? fabs(d2 / dref - 1.0) : 0.0);   /* |S11|-only jobs: D cancels in the ratio */
                } else {
                    const double got = std::norm(P_ + hp->rs * Q_) / d2, ref = std::norm(a + hp->rs * b);
                    rel = need_s21 ? fabs(got - ref) / ref : 0.0;
                    if (gd) {
                        /* group delay: the derivative polynomials against the central difference of the per-element chain's phase
                         * over x (1 +- 1e-6) -- the definition the sweep API and the oracle use */
                        cplx Np(0, 0), Dp(0, 0);
                        const cplx sj1(0.0, x);
                        cplx pw(1.0, 0.0);
                        for (int i = 1; i < 2 * kn; i++) { Np += (double)i * (c.pp[i] + hp->rs * zni * c.qq[i]) * pw; pw *= sj1; }
                        pw = cplx(1.0, 0.0);
                        for (int i = 1; i < 2 * out->kd && out->den == QO_TF_DEN_DD; i++) { Dp += (double)i * c.dd[i] * pw; pw *= sj1; }
                        const cplx Nn = P_ + hp->rs * Q_;
                        double tau = (Np / Nn).real();
                        if (out->den == QO_TF_DEN_DD) tau -= (Dp / tf_horner_host(c.dd, out->kd, x)).real();
                        cplx dv[2];
                        for (int sgn = 0; sgn < 2; sgn++) {
                            const double xq = x * (sgn ? 1.0 - 1e-6 : 1.0 + 1e-6), yq = -xq * xq;
                            double ar2 = hp->rl, ai2 = 0.0, br2 = 1.0, bi2 = 0.0;
                            for (int e = nl - 1; e >= 0; e--) {
                                const double *nd = c.nd[e];
                                const double nr = nd[2] * yq + nd[0], ni = nd[1] * xq, dr = nd[5] * yq + nd[3], di = nd[4] * xq;
                                const double inv = 1.0 / (dr * dr + di * di);
                                const double ir = (nr * dr + ni * di) * inv, ii = (ni * dr - nr * di) * inv;
                                if (c.ser[e]) { const double tr = ir * br2 - ii * bi2, ti = ir * bi2 + ii * br2; ar2 += tr; ai2 += ti; }
                                else { const double tr = ir * ar2 - ii * ai2, ti = ir * ai2 + ii * ar2; br2 += tr; bi2 += ti; }
                            }
                            dv[sgn] = cplx(ar2 + hp->rs * br2, ai2 + hp->rs * bi2);
                        }
                        const cplx cr = dv[0] * std::conj(dv[1]);
                        const double tau_fd = atan2(cr.imag(), cr.real()) / (2e-6 * x);
                        /* the finite difference itself carries ~1e-10 of rounding noise relative to the largest delay; 1e-7 is far below any spec resolution */
                        const double egd = 1e-3 * fabs(tau - tau_fd) / (fabs(tau_fd) > 1e-3 ? fabs(tau_fd) : 1e-3);
                        if (egd > rel) rel = egd;
                    }
                    if (s11) {
                        /* |S11|^2, relative with an absolute floor of -40 dB (return-loss nulls are not thresholds) */
                        const double g11 = std::norm(P_ - hp->rs * Q_) / std::norm(P_ + hp->rs * Q_), r11 = std::norm(a - hp->rs * b) / ref;
                        const double e11 = fabs(g11 - r11) / (r11 > 1e-4 ? r11 : 1e-4);
                        if (e11 > rel) rel = e11;
                    }
                }
                if (!(rel == rel)) rel = 1e300;
                if (rel > worst) worst = rel;
            }
        }
        accepted = range_ok && worst <= tol;
    }
    out->err = worst;
    if (!accepted) QO_TF_NO("polynomial expansion is too ill-conditioned on this grid");
    tf_fuse_gate(hp, nf, xg.data(), mask, cs, zni, out);
    out->reason = "ok";
    return 1;
#undef QO_TF_NO
}


/* ---- FULL_S flavour (qo_tf_fs.cuh) --------------------------------------------------------------------------- */
extern "C" int qo_tf_fs_launch(int dmode, int sm_count, const TfFsParams *P, cudaStream_t st)
{
    const int tpb = 128, minb = 4;
    const unsigned long long warps = tpb / 32;
    unsigned long long blocks = (P->nsamples + warps - 1) / warps;
    const unsigned long long resident = (unsigned long long)sm_count * minb;
    if (blocks > resident) blocks = resident;
    if (blocks < 1) blocks = 1;
    if (dmode == 2) qo_fs_tf_kernel<2, 2, 128, 4><<<(unsigned)blocks, tpb, 0, st>>>(*P);
    else if (dmode == 1) qo_fs_tf_kernel<1, 2, 128, 4><<<(unsigned)blocks, tpb, 0, st>>>(*P);
    else qo_fs_tf_kernel<0, 2, 128, 4><<<(unsigned)blocks, tpb, 0, st>>>(*P);
    return (int)cudaGetLastError();
}

/* Can FULL_S launches of this job run on qo_fs_tf_kernel?  Lumped cascade, no coupler; polynomial lengths by the same
 * tail rule; self-check of S11, S21, S22 (complex) against the per-element ABCD chain at the nominal network (every
 * point) and both ends of the tolerance box (every 4th point). */
extern "C" int qo_tf_fs_plan_check(const DevProg *hp, int mode_full_s, int precision, int generic, const double *f, int nf, const QoOverrides *ov,
                                   TfPlan *out)
{
    memset(out, 0, sizeof *out);
    out->cpl_op = -1;
#define QO_TF_NO(msg) do { out->reason = msg; return 0; } while (0)
    if (ov->kernel == QoOverrides::INTERP || ov->kernel == QoOverrides::LADDER) QO_TF_NO("QO100NET_KERNEL override");
    if (generic || !mode_full_s || precision != 64) QO_TF_NO("not an FP64 FULL_S job on a lumped cascade");
    const int e0 = hp->op0, nl = hp->n_ops - e0;
    if (nl < 1 || nl > QO_TF_MAXEL || hp->n_var > QO_MAX_VAR) QO_TF_NO("element count");
    int deg = 0, has_d = 0;
    for (int e = 0; e < nl; e++) {
        const int op = hp->opcode[e0 + e], dg = qo_tf_degree(op);
        if (dg < 0) QO_TF_NO("non-lumped element");
        deg += dg;
        if (!(op == OP_SER_R || op == OP_SER_L || op == OP_SHUNT_C)) has_d = 1;
    }
    if (deg > 2 * QO_TF_MAXK - 1) QO_TF_NO("polynomial degree");
    const int Kfull = deg / 2 + 1;
    out->deg = deg; out->el0 = e0; out->n_el = nl; out->nn = 6; out->den = has_d ? QO_TF_DEN_D : QO_TF_DEN_NONE;
    const double two_pi = 6.283185307179586476925286766559;
    double f_lo = f[0], f_hi = f[0];
    for (int k = 1; k < nf; k++) { if (f[k] < f_lo) f_lo = f[k]; if (f[k] > f_hi) f_hi = f[k]; }
    const double wr = two_pi * sqrt(f_lo * f_hi);
    out->wref = wr;
    const double rs = hp->rs, rl = hp->rl, zn = sqrt(rs * rl), zni = 1.0 / zn, k21 = hp->k21;
    const double trunc = ov->tf_trunc, tol = ov->tf_tol;
    const int NCORN = hp->n_var > 0 ? QO_TF_NCORNER : 2;
    std::vector<TfCorner> cs((size_t)NCORN), c2((size_t)NCORN);
    for (int ci = 0; ci < NCORN; ci++) {
        TfCorner &c = cs[ci];
        double xv[QO_MAX_VAR];
        tf_corner_vars(hp, e0, nl, ci, xv);
        for (int e = 0; e < nl; e++) {
            double p[6];
            for (int k = 0; k < 6; k++) {
                p[k] = hp->nom[e0 + e][k];
                if (hp->tvar[e0 + e][k] >= 0) p[k] = qo_stream_apply(p[k], hp->ttol[e0 + e][k], xv[hp->tvar[e0 + e][k]], hp->tmode[e0 + e][k]);
            }
            c.ser[e] = qo_tf_element(hp->opcode[e0 + e], p, wr, c.nd[e]);
            const double sc = c.ser[e] ? zni : zn;
            const double *nd = c.nd[e];
            double *rec = c.rec[e];
            rec[0] = nd[0] * sc; rec[1] = nd[1] * sc; rec[2] = nd[2] * sc; rec[3] = nd[3]; rec[4] = nd[4]; rec[5] = nd[5];
            rec[6] = 1.0; rec[7] = 0.0; rec[8] = 0.0; rec[9] = c.ser[e] ? 1.0 : 0.0;
        }
        c2[ci] = c;
        tf_expand_host(c.rec, nl, rl, zn, c.pp, c.qq, c.dd, c.ee);
        tf_expand_host(c2[ci].rec, nl, -rl, zn, c2[ci].pp, c2[ci].qq, c2[ci].dd, c2[ci].ee);
    }
    /* kept lengths: terms that stay below `trunc` of |P| + zn |Q| (numerators) / |D| everywhere on the grid */
    const int NC = 2 * Kfull;
    int kn = 1, kdd = 1;
    std::vector<double> xpw((size_t)NC + 1);
    for (int k = 0; k < nf; k++) {
        const double x = two_pi * f[k] / wr;
        xpw[0] = 1.0; for (int i = 1; i <= NC; i++) xpw[i] = xpw[i - 1] * x;
        for (int ci = 0; ci < NCORN; ci++) {
            if (ci > 2 && (k & 3) && k + 1 < nf) continue;
            for (int which = 0; which < 2; which++) {
                const TfCorner &c = which ? c2[ci] : cs[ci];
                const double nref = trunc * (sqrt(std::norm(tf_horner_host(c.pp, Kfull, x))) + sqrt(std::norm(tf_horner_host(c.qq, Kfull, x))));
                double acc = 0.0;
                int K = Kfull;
                while (K > kn) {
                    acc += (fabs(c.pp[2 * K - 1]) + fabs(c.qq[2 * K - 1])) * xpw[2 * K - 1] + (fabs(c.pp[2 * K - 2]) + fabs(c.qq[2 * K - 2])) * xpw[2 * K - 2];
                    if (acc > nref) break;
                    K--;
                }
                if (K > kn) kn = K;
            }
            if (has_d) {
                const TfCorner &c = cs[ci];
                const double dref = trunc * sqrt(std::norm(tf_horner_host(c.dd, Kfull, x)));
                double acc = 0.0;
                int K = Kfull;
                while (K > kdd) { acc += fabs(c.dd[2 * K - 1]) * xpw[2 * K - 1] + fabs(c.dd[2 * K - 2]) * xpw[2 * K - 2]; if (acc > dref) break; K--; }
                if (K > kdd) kdd = K;
            }
        }
    }
    out->kn = kn; out->kd = has_d ? kdd : 0;
    /* a branch that resonates inside the grid (trap / tank, Q > 5): D as the product of the branch denominators (qo_tf_fs.cuh) */
    int factored = 0;
    if (has_d) {
        const double xlo = two_pi * f_lo / wr * 0.8, xhi = two_pi * f_hi / wr * 1.25;
        for (int e = 0; e < nl; e++) {
            const double *nd = cs[1].nd[e];
            if (nd[3] > 0.0 && nd[5] > 0.0 && nd[4] * nd[4] < 0.04 * nd[3] * nd[5]) {
                const double xr = sqrt(nd[3] / nd[5]);
                if (xr > xlo && xr < xhi) factored = 1;
            }
        }
    }
    if (factored) { out->den = QO_TF_DEN_E + 100; out->kd = 0; }          /* marker: factored D (launch_tf_fs reads it) */
    /* self-check: S11, S21, S22 from the kept polynomials against the per-element ABCD chain */
    double worst = 0.0;
    for (int ci = 0; ci < NCORN; ci++) {
        const TfCorner &c = cs[ci], &cb = c2[ci];
        for (int k = 0; k < nf; k++) {
            if (ci != QO_TF_NOMINAL && (k & 3) && k > 0 && k + 1 < nf) continue;
            const double x = two_pi * f[k] / wr, y = -x * x;
            const cplx Pv = tf_horner_host(c.pp, kn, x), Qv = tf_horner_host(c.qq, kn, x) * zni;
            const cplx P2 = tf_horner_host(cb.pp, kn, x), Q2 = tf_horner_host(cb.qq, kn, x) * zni;
            cplx Dv = has_d ? tf_horner_host(c.dd, kdd, x) : cplx(1.0, 0.0);
            if (factored) { Dv = cplx(1.0, 0.0); for (int e = 0; e < nl; e++) Dv *= cplx(c.nd[e][5] * y + c.nd[e][3], c.nd[e][4] * x); }
            const cplx num = Pv + rs * Qv;
            const cplx g21 = k21 * Dv / num, g11 = (Pv - rs * Qv) / num, g22 = (P2 + rs * Q2) / num;
            cplx A(1, 0), B(0, 0), C(0, 0), Dd(1, 0);
            for (int e = 0; e < nl; e++) {
                const double *nd = c.nd[e];
                const cplx N(nd[2] * y + nd[0], nd[1] * x), De(nd[5] * y + nd[3], nd[4] * x);
                const cplx imm = N / De;
                if (c.ser[e]) { B += A * imm; Dd += C * imm; } else { A += B * imm; C += Dd * imm; }
            }
            const cplx den = A * rl + B + rs * (C * rl + Dd);
            const cplx r21 = k21 / den, r11 = (A * rl + B - rs * (C * rl + Dd)) / den, r22 = (-A * rl + B - rs * C * rl + rs * Dd) / den;
            double rel = std::abs(g21 - r21) / std::abs(r21);
            const double e11 = std::abs(g11 - r11) / fmax(std::abs(r11), 0.02), e22 = std::abs(g22 - r22) / fmax(std::abs(r22), 0.02);
            if (e11 > rel) rel = e11;
            if (e22 > rel) rel = e22;
            if (!(rel == rel)) rel = 1e300;
            if (rel > worst) worst = rel;
        }
    }
    out->err = worst;
    if (worst > tol) QO_TF_NO("polynomial expansion is too ill-conditioned on this grid");
    out->reason = "ok";
    return 1;
#undef QO_TF_NO
}
