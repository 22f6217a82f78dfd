/*
 * qo_nodal.cu -- N-port nodal analysis on the GPU (SURVEY row N4), sm_100a.
 *
 * Replaces qucsator's S-parameter analysis for networks that are not a cascade: the reference's bias networks
 * util/pa-bias-simulation/pa-bias-simulation.sch:19-72 (result: pa-bias-simulation.dat:1-85035).
 *
 * One thread owns one (sample, frequency) point: it stamps the modified-nodal matrix A (node voltages plus
 * one branch current per VCVS; port terminations 1/Z_k included), factorises it in place (LU, partial
 * pivoting) and back-substitutes once per port:  S[k][j] = 2 sqrt(Z_j/Z_k) V_k - delta_kj  with 1/Z_j
 * injected at port j.  A lives in thread-local memory (the hardware interleaves it across the warp, so a
 * warp's accesses to "its" element (i,j) are coalesced and L1-resident); its leading dimension is a template
 * parameter so that small networks do not pay for the largest.  Per sample the block first derives the
 * perturbed branch parameters (the shared bit-exact Philox stream) into shared memory.  Measured two-port
 * blocks carry no tolerances: their 2x2 admittance per grid point is tabulated on the host at plan time with
 * the same SPfile interpolation the cascade path uses.
 *
 * Work per point ~ (8/3) n^3 real FMAs (n = unknowns): FP64-bound, no reuse across points -- like the cascade
 * kernels this is latency/FP64-pipe bound, not memory bound.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <memory>
#include <vector>

#include "qo_ctx_internal.h"
#include "qo_overrides.h"
#include "qo_stream.h"

#include "qo_nodal_prog.h"

__device__ __forceinline__ double2 c_mul(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ double2 c_sub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ double2 c_add(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 c_inv(double2 b) { const double d = 1.0 / (b.x * b.x + b.y * b.y); return make_double2(b.x * d, -b.y * d); }
/* a -= l * u (complex fused multiply-subtract, 4 DFMA) */
__device__ __forceinline__ double2 c_fms(double2 a, double2 l, double2 u)
{
    a.x = fma(-l.x, u.x, a.x); a.x = fma(l.y, u.y, a.x);
    a.y = fma(-l.x, u.y, a.y); a.y = fma(-l.y, u.x, a.y);
    return a;
}

/* ---- static (symbolic) factorisation plan ----------------------------------------------------------------
 * Every point of a job has the same sparsity pattern, and for these networks the same pivot order works over
 * the whole band, so the host factorises ONCE symbolically: it takes the row order a pivoted LU chooses at a
 * representative point, computes the fill pattern, packs the non-zeros (fill included) into a compact value
 * array and emits a branch-free "program" of value-array indices for elimination and substitutions.  The
 * kernel then runs that program -- no pivot search, no row swaps, no zero tests, ~10x fewer value accesses than
 * the dense factorisation.  The host runs the same program at several grid points and compares with the
 * pivoted dense solution; if they disagree (a pivot that is only good at some frequencies) the job falls back
 * to the dense kernel (QO100NET_NODAL=dense forces it). */
#define QN_PROG_MAX 6144       /* uint16 words of program */
#define QN_NNZ_MAX 512
struct NodalStatic {
    int32_t n, nnz, prog_len, stamp_at, zero_at, n_zero;   /* stamp stream / fill-only value indices inside prog[] */
    int32_t solve_at[QO_NODAL_MAX_PORTS];               /* start of each port's pruned substitution program */
    int16_t pos[QO_NODAL_MAX_UNK * QO_NODAL_MAX_UNK];   /* (pivot-order row, permuted column) -> value index, -1 = structural zero */
    uint8_t rowmap[QO_NODAL_MAX_UNK];                   /* original row (equation) -> pivot-order row */
    uint8_t colmap[QO_NODAL_MAX_UNK];                   /* original unknown -> permuted column (port unknowns last) */
    uint16_t prog[QN_PROG_MAX];
    double worst_l2;                                    /* largest |multiplier|^2 the plan-time probes met */
};

/* where a stamp lands: a dense matrix with leading dimension LD (dense kernel, host analysis) ... */
template <int LD> struct DenseSink {
    double2 *A;
    __host__ __device__ __forceinline__ void add(int r, int c, double2 v) { A[r * LD + c].x += v.x; A[r * LD + c].y += v.y; }
};
/* ... or the compact value array of the static plan.  The order of the add() calls of nodal_stamp_all depends only on the netlist, so the host records, once per
 * job, the value index every call lands on (bit 15: first touch -> store instead of add); the kernel replays
 * that stream and never looks at (row, column) again: no index tables, no zero-fill of stamped values. */
struct ReplaySink {
    double2 *V;
    const uint16_t *st;
    int k;
    __host__ __device__ __forceinline__ void add(int, int, double2 v)
    {
        const unsigned int wd = st[k++];
        const int q = (int)(wd & 0x7fffu);
        if (wd >> 15) V[q] = v;
        else { V[q].x += v.x; V[q].y += v.y; }
    }
};

template <class Sink> __host__ __device__ __forceinline__ void stamp_y(Sink &S, int a, int b, double2 y)
{
    const double2 my = make_double2(-y.x, -y.y);
    if (a) S.add(a - 1, a - 1, y);
    if (b) S.add(b - 1, b - 1, y);
    if (a && b) { S.add(a - 1, b - 1, my); S.add(b - 1, a - 1, my); }
}

__host__ __device__ __forceinline__ double2 hd_mul(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__host__ __device__ __forceinline__ double2 hd_inv(double2 b) { const double d = 1.0 / (b.x * b.x + b.y * b.y); return make_double2(b.x * d, -b.y * d); }
__host__ __device__ __forceinline__ double2 hd_fms(double2 a, double2 l, double2 u)
{
    a.x = fma(-l.x, u.x, a.x); a.x = fma(l.y, u.y, a.x);
    a.y = fma(-l.x, u.y, a.y); a.y = fma(-l.y, u.x, a.y);
    return a;
}

/* all stamps of one (sample, frequency) point: branches with the sample's parameters par[b][0..3], the measured
 * blocks' tabulated admittances yk (4 values per block branch, in branch order), port terminations */
template <class Sink>
__host__ __device__ __forceinline__ void nodal_stamp_all(const NodalProg *prog, const double (*par)[4], double w, const double2 *yk,
                                                         size_t yk_stride, Sink &S)
{
    int extra = prog->n_nodes, iblk = 0;
    for (int b = 0; b < prog->nb; b++) {
        const int kind = prog->kind[b];
        const int n0 = prog->node[b][0], n1 = prog->node[b][1], n2 = prog->node[b][2], n3 = prog->node[b][3];
        const double p0 = par[b][0], p1 = par[b][1], p2 = par[b][2];
        if (kind == QO_NB_R) stamp_y(S, n0, n1, make_double2(1.0 / p0, 0.0));
        else if (kind == QO_NB_L) {                /* Y = (1 - w^2 L Cp + j w R Cp) / (R + jwL) */
            const double2 num = make_double2(1.0 - w * w * p0 * p2, w * p1 * p2);
            stamp_y(S, n0, n1, hd_mul(num, hd_inv(make_double2(p1, w * p0))));
        } else if (kind == QO_NB_C) {              /* Y = 1 / (R + j(w Ls - 1/(wC))) */
            stamp_y(S, n0, n1, hd_inv(make_double2(p1, w * p2 - 1.0 / (w * p0))));
        } else if (kind == QO_NB_VCVS) {           /* in+ n0, out+ n1, out- n2, in- n3; current unknown kx */
            const int kx = extra++;
            const double cs = cos(w * p1), sn = sin(w * p1);
            const double2 g = make_double2(p0 * cs, -p0 * sn), mg = make_double2(-g.x, -g.y);
            const double2 one = make_double2(1.0, 0.0), mone = make_double2(-1.0, 0.0);
            if (n1) { S.add(n1 - 1, kx, one); S.add(kx, n1 - 1, one); }
            if (n2) { S.add(n2 - 1, kx, mone); S.add(kx, n2 - 1, mone); }
            if (n0) S.add(kx, n0 - 1, mg);
            if (n3) S.add(kx, n3 - 1, g);
        } else if (kind == QO_NB_SBLOCK) {         /* tabulated 2x2 admittance; indefinite form with reference n2 */
            const double2 *y = yk + (size_t)iblk * yk_stride;
            iblk++;
            const int t[3] = { n0, n1, n2 };
            double2 Y3[3][3];
            Y3[0][0] = y[0]; Y3[0][1] = y[1]; Y3[1][0] = y[2]; Y3[1][1] = y[3];
            Y3[0][2] = make_double2(-(y[0].x + y[1].x), -(y[0].y + y[1].y));
            Y3[1][2] = make_double2(-(y[2].x + y[3].x), -(y[2].y + y[3].y));
            for (int c = 0; c < 3; c++) Y3[2][c] = make_double2(-(Y3[0][c].x + Y3[1][c].x), -(Y3[0][c].y + Y3[1][c].y));
            for (int r = 0; r < 3; r++)
                for (int c = 0; c < 3; c++)
                    if (t[r] && t[c]) S.add(t[r] - 1, t[c] - 1, Y3[r][c]);
        }
    }
    for (int p = 0; p < prog->np; p++) S.add(prog->port_node[p] - 1, prog->port_node[p] - 1, make_double2(1.0 / prog->port_z0[p], 0.0));
}

/* run the elimination part of a static program on the value array V.  Returns the largest |multiplier|^2 met: per-point
 * partial pivoting keeps every multiplier <= 1; the fixed order does not, and a huge one means this point (this sample's
 * values at this frequency) wanted another pivot -- the caller counts such points and the host re-runs the job on the
 * pivoted dense kernel (QN_GROWTH2) */
__host__ __device__ __forceinline__ double static_factor(const uint16_t *pg, int n, double2 *V)
{
    double lmax2 = 0.0;
    int ip = 0;
    for (int c = 0; c < n; c++) {
        const int nu = pg[ip + 1];
        const uint16_t *ucol = pg + ip + 2;          /* value indices of the pivot row's entries right of the pivot */
        const int nrows = pg[ip + 2 + nu];
        if (nrows == 0) { ip += 3 + nu; continue; }  /* nothing below the pivot */
        const double2 inv = hd_inv(V[pg[ip]]);
        ip += 3 + nu;
        for (int r = 0; r < nrows; r++) {
            const int prc = pg[ip++];
            const double2 l = hd_mul(V[prc], inv);
            V[prc] = l;
            const double l2 = fma(l.x, l.x, l.y * l.y);
            lmax2 = !(l2 <= lmax2) ? l2 : lmax2;                       /* NaN sticks */
            for (int q = 0; q < nu; q++) { const int prj = pg[ip + q]; V[prj] = hd_fms(V[prj], l, V[ucol[q]]); }
            ip += nu;
        }
    }
    return lmax2;
}
/* |multiplier| above 3e6 or NaN: the point is suspect.  Rounding errors are amplified by at most the multiplier, so 3e6 x
 * 1.1e-16 = 3e-10 stays inside the 1e-9 parity bar; the reference's stiff bias network (100 uF next to 1.2 pF) legitimately
 * reaches 3e5 at 1 MHz under its ports-last order and still matches the reference dataset, a vanishing pivot gives >= 1e15 */
#define QN_GROWTH2 1e13

/* One port's substitutions, pruned symbolically: the program lists only the rows the unit right-hand side can
 * reach (forward) and only the rows the port unknowns depend on (backward).  Stream at `at`:
 *   n_fwd, { row i, n_terms, { q, value index } ... } ...,  n_bwd, { row i, diag index, n_terms, { q, value index } ... } ...
 * x must be zero except for the injected entry. */
__host__ __device__ __forceinline__ void static_solve(const uint16_t *pg, int at, const double2 *V, double2 *x)
{
    int ip = at;
    const int nfwd = pg[ip++];
    for (int t = 0; t < nfwd; t++) {
        const int i = pg[ip++], nl = pg[ip++];
        double2 acc = x[i];
        for (int q = 0; q < nl; q++) { acc = hd_fms(acc, V[pg[ip + 1]], x[pg[ip]]); ip += 2; }
        x[i] = acc;
    }
    const int nbwd = pg[ip++];
    for (int t = 0; t < nbwd; t++) {
        const int i = pg[ip++], pii = pg[ip++], nu = pg[ip++];
        double2 acc = x[i];
        for (int q = 0; q < nu; q++) { acc = hd_fms(acc, V[pg[ip + 1]], x[pg[ip]]); ip += 2; }
        x[i] = hd_mul(acc, hd_inv(V[pii]));
    }
}

/*
 * unit u = sample * nchunks + chunk; a block works on one unit at a time: QN_TPB consecutive grid points per
 * pass.  Reduce-only jobs use nchunks == 1 (the block walks the whole grid of its sample and then reduces).
 */
/* MODE 0: dense, per-point pivoting | 1: static plan, values in a private (local-memory) array of NNZ entries */
template <int LD, int MODE, int NNZ>
__global__ void __launch_bounds__(QN_TPB)
qo_nodal_kernel(const NodalProg *__restrict__ prog, const NodalStatic *__restrict__ splan, const double *__restrict__ fgrid,
                const unsigned char *__restrict__ mask, const double2 *__restrict__ yblk, int nf, int chunk_len, int nchunks,
                unsigned long long sample_offset, unsigned long long nsamples, unsigned long long *__restrict__ counters,
                double2 *__restrict__ s_out, double growth2)
{
    /* static plan staged in shared memory: every thread walks the same program (broadcast reads) */
    constexpr bool STATIC = MODE != 0;
    __shared__ uint8_t s_rowmap[QO_NODAL_MAX_UNK], s_colmap[QO_NODAL_MAX_UNK];
    __shared__ uint16_t s_prog[STATIC ? QN_PROG_MAX : 1];
    if (STATIC) {
        for (int i = threadIdx.x; i < QO_NODAL_MAX_UNK; i += QN_TPB) { s_rowmap[i] = splan->rowmap[i]; s_colmap[i] = splan->colmap[i]; }
        for (int i = threadIdx.x; i < splan->prog_len; i += QN_TPB) s_prog[i] = splan->prog[i];
    }
    __shared__ double s_p[QO_NODAL_MAX_BR][4];
    __shared__ double s_x[QN_MAX_VAR];
    __shared__ double s_trk[QN_MAX_SPEC][QN_TPB / 32];
    __shared__ unsigned int s_cnt[2 + QN_MAX_SPEC + 1024];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = prog->n_unk, np = prog->np, nb = prog->nb, nspec = prog->nspec, n_nodes = prog->n_nodes;
    const int full = prog->full;
    const int ncnt = 2 + nspec + (prog->hist_bins > 0 ? prog->hist_bins : 0);
    for (int i = tid; i < ncnt; i += QN_TPB) s_cnt[i] = 0;
    unsigned int n_suspect = 0;                      /* points whose fixed pivot order met a huge multiplier (static plan) */
    __syncthreads();

    const unsigned long long n_units = nsamples * (unsigned long long)nchunks;
    for (unsigned long long u = blockIdx.x; u < n_units; u += gridDim.x) {
        const unsigned long long s = u / (unsigned long long)nchunks;
        const int chunk = (int)(u - s * (unsigned long long)nchunks);
        /* per-sample branch parameters */
        for (int v = tid; v < prog->n_var; v += QN_TPB) s_x[v] = qo_stream_variate(prog->seed, sample_offset + s, (uint32_t)v, prog->dist);
        __syncthreads();
        for (int i = tid; i < nb * 4; i += QN_TPB) {
            const int b = i >> 2, k = i & 3;
            double v = prog->nom[b][k];
            const int tv = prog->tvar[b][k];
            if (tv >= 0) v = qo_stream_apply(v, prog->ttol[b][k], s_x[tv], prog->tmode[b][k]);
            s_p[b][k] = v;
        }
        __syncthreads();

        double trk[QN_MAX_SPEC];
#pragma unroll
        for (int sp = 0; sp < QN_MAX_SPEC; sp++) trk[sp] = -1e300;       /* running max of (+-)|S|^2 */
        const int k_lo = chunk * chunk_len, k_hi = min(nf, k_lo + chunk_len);
        for (int k = k_lo + tid; k < k_hi; k += QN_TPB) {
            const double w = 6.283185307179586476925286766559 * fgrid[k];
            const double2 *yk = yblk + (size_t)k * 4;                 /* block admittances: [block][nf][4] */
            double2 A[STATIC ? NNZ : LD * LD];
            int perm[STATIC ? 1 : LD];
            unsigned int lmask[STATIC ? 1 : LD], umask[STATIC ? 1 : LD];
            bool singular = false;
            if (STATIC) {
                for (int i = 0; i < splan->n_zero; i++) A[s_prog[splan->zero_at + i]] = make_double2(0.0, 0.0);   /* fill-only */
                ReplaySink S = { A, s_prog + splan->stamp_at, 0 };
                nodal_stamp_all(prog, s_p, w, yk, (size_t)nf * 4, S);
                const double l2 = static_factor(s_prog, n, A);
                if (!(l2 <= growth2)) n_suspect++;
            } else {
                for (int i = 0; i < n; i++) {
                    perm[i] = i;
                    for (int j = 0; j < n; j++) A[i * LD + j] = make_double2(0.0, 0.0);
                }
                DenseSink<LD> S = { A };
                nodal_stamp_all(prog, s_p, w, yk, (size_t)nf * 4, S);
                /* LU, partial pivoting (rows are swapped physically: n <= 32), walking bit masks of the non-zero
                 * columns instead of full rows; lmask/umask record the factors' patterns for the substitutions */
                for (int c = 0; c < n; c++) {
                    int piv = c;
                    double best = A[c * LD + c].x * A[c * LD + c].x + A[c * LD + c].y * A[c * LD + c].y;
                    for (int r = c + 1; r < n; r++) {
                        const double2 v = A[r * LD + c];
                        const double m = v.x * v.x + v.y * v.y;
                        if (m > best) { best = m; piv = r; }
                    }
                    if (!(best > 0.0)) { singular = true; break; }
                    if (piv != c) {
                        for (int j = 0; j < n; j++) { const double2 t = A[c * LD + j]; A[c * LD + j] = A[piv * LD + j]; A[piv * LD + j] = t; }
                        const int t = perm[c]; perm[c] = perm[piv]; perm[piv] = t;
                    }
                    unsigned int nz = 0;
                    for (int j = c + 1; j < n; j++) { const double2 v = A[c * LD + j]; if (v.x != 0.0 || v.y != 0.0) nz |= 1u << j; }
                    umask[c] = nz;
                    const double2 inv = c_inv(A[c * LD + c]);
                    for (int r = c + 1; r < n; r++) {
                        const double2 a = A[r * LD + c];
                        if (a.x == 0.0 && a.y == 0.0) continue;
                        const double2 l = c_mul(a, inv);
                        A[r * LD + c] = l;
                        for (unsigned int m = nz; m; m &= m - 1) {
                            const int j = __ffs((int)m) - 1;
                            A[r * LD + j] = c_fms(A[r * LD + j], l, A[c * LD + j]);
                        }
                    }
                }
                if (!singular)
                    for (int i = 0; i < n; i++) {
                        unsigned int lm = 0;
                        for (int q = 0; q < i; q++) { const double2 v = A[i * LD + q]; if (v.x != 0.0 || v.y != 0.0) lm |= 1u << q; }
                        lmask[i] = lm;
                    }
            }
            const size_t obase = (((size_t)s * (size_t)nf + (size_t)k) * (size_t)np) * (size_t)np;
            const unsigned int mb = mask[k];
            for (int j = 0; j < np; j++) {
                double2 x[LD];
                const int src = prog->port_node[j] - 1;
                if (STATIC) {
                    for (int i = 0; i < n; i++) x[i] = make_double2(0.0, 0.0);
                    x[s_rowmap[src]] = make_double2(1.0 / prog->port_z0[j], 0.0);
                    static_solve(s_prog, splan->solve_at[j], A, x);
                } else {
                    for (int i = 0; i < n; i++) x[i] = make_double2(perm[i] == src ? 1.0 / prog->port_z0[j] : 0.0, 0.0);
                    if (singular) { for (int i = 0; i < n; i++) x[i] = make_double2(nan(""), nan("")); }
                    else {
                        for (int i = 1; i < n; i++) {
                            double2 acc = x[i];
                            for (unsigned int m = lmask[i]; m; m &= m - 1) { const int q = __ffs((int)m) - 1; acc = c_fms(acc, A[i * LD + q], x[q]); }
                            x[i] = acc;
                        }
                        for (int i = n - 1; i >= 0; i--) {
                            double2 acc = x[i];
                            for (unsigned int m = umask[i]; m; m &= m - 1) { const int q = __ffs((int)m) - 1; acc = c_fms(acc, A[i * LD + q], x[q]); }
                            x[i] = c_mul(acc, c_inv(A[i * LD + i]));
                        }
                    }
                }
                for (int kk = 0; kk < np; kk++) {
                    const double sc = 2.0 * sqrt(prog->port_z0[j] / prog->port_z0[kk]);
                    const double2 v = x[STATIC ? s_colmap[prog->port_node[kk] - 1] : prog->port_node[kk] - 1];
                    const double2 sv = make_double2(sc * v.x - (kk == j ? 1.0 : 0.0), sc * v.y);
                    if (full) s_out[obase + (size_t)kk * np + j] = sv;
#pragma unroll
                    for (int sp = 0; sp < QN_MAX_SPEC; sp++)
                        if (sp < nspec && ((mb >> sp) & 1u) && prog->spec_row[sp] == kk && prog->spec_col[sp] == j) {
                            const double m2 = sv.x * sv.x + sv.y * sv.y;
                            const double c = prog->spec_min[sp] ? -m2 : m2;
                            if (c > trk[sp] || m2 != m2) trk[sp] = m2 != m2 ? 1e300 : c;
                        }
                }
            }
        }
        if (!full) {
            /* per-sample verdict: block max of every tracker */
#pragma unroll
            for (int sp = 0; sp < QN_MAX_SPEC; sp++) {
                if (sp < nspec) {
                    double v = trk[sp];
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) { const double o = __shfl_xor_sync(0xffffffffu, v, off); v = o > v ? o : v; }
                    if (lane == 0) s_trk[sp][warp] = v;
                }
            }
            __syncthreads();
            if (tid == 0) {
                unsigned int fail = 0;
                double hist_worst = 0.0;
                for (int sp = 0; sp < nspec; sp++) {
                    double v = s_trk[sp][0];
                    for (int q = 1; q < QN_TPB / 32; q++) v = s_trk[sp][q] > v ? s_trk[sp][q] : v;
                    if (v == -1e300) continue;                          /* the spec covers no grid point */
                    const double thr = prog->spec_min[sp] ? -prog->spec_thr[sp] : prog->spec_thr[sp];
                    if (v > thr) fail |= 1u << sp;
                    if (sp == prog->hist_spec) hist_worst = fabs(v);
                }
                atomicAdd(&s_cnt[0], fail == 0 ? 1u : 0u);
                atomicAdd(&s_cnt[1], 1u);
                for (int sp = 0; sp < nspec; sp++) if ((fail >> sp) & 1u) atomicAdd(&s_cnt[2 + sp], 1u);
                if (prog->hist_bins > 0) {
                    const double v = 10.0 * log10(hist_worst);
                    const double xb = (v - prog->hist_lo) / (prog->hist_hi - prog->hist_lo) * (double)prog->hist_bins;
                    long long b = (long long)floor(xb);
                    if (!(xb >= 0.0)) b = 0;
                    if (b >= prog->hist_bins) b = prog->hist_bins - 1;
                    atomicAdd(&s_cnt[2 + nspec + (int)b], 1u);
                }
            }
        }
        __syncthreads();
    }
    if (!full) {
        for (int i = tid; i < ncnt; i += QN_TPB)
            if (s_cnt[i]) atomicAdd(&counters[i], (unsigned long long)s_cnt[i]);
    }
    if (STATIC && n_suspect) atomicAdd(&counters[ncnt], (unsigned long long)n_suspect);     /* one slot past the job's counters */
}

/* ---- host side ------------------------------------------------------------------------------------------ */
static qo_c64 h_mul(qo_c64 a, qo_c64 b) { qo_c64 r = { a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re }; return r; }
static qo_c64 h_div(qo_c64 a, qo_c64 b)
{
    const double d = b.re * b.re + b.im * b.im;
    qo_c64 r = { (a.re * b.re + a.im * b.im) / d, (a.im * b.re - a.re * b.im) / d };
    return r;
}

/* 2x2 admittance of a measured block: Y = (I - S)(I + S)^-1 / z0; y = { y11, y12, y21, y22 } */
static void s_to_y(const qo_c64 s[4], double z0, qo_c64 y[4])
{
    const qo_c64 s11 = s[0], s21 = s[1], s12 = s[2], s22 = s[3];
    const qo_c64 a = { 1.0 + s11.re, s11.im }, d = { 1.0 + s22.re, s22.im }, m11 = { 1.0 - s11.re, -s11.im }, m22 = { 1.0 - s22.re, -s22.im };
    const qo_c64 p = h_mul(s12, s21), ad = h_mul(a, d), det = { ad.re - p.re, ad.im - p.im };
    qo_c64 t, u;
    t = h_mul(m11, d); t.re += p.re; t.im += p.im; y[0] = h_div(t, det);
    t = h_mul(s12, a); u = h_mul(m11, s12); t.re = -t.re - u.re; t.im = -t.im - u.im; y[1] = h_div(t, det);
    t = h_mul(s21, d); u = h_mul(m22, s21); t.re = -t.re - u.re; t.im = -t.im - u.im; y[2] = h_div(t, det);
    t = h_mul(m22, a); t.re += p.re; t.im += p.im; y[3] = h_div(t, det);
    for (int i = 0; i < 4; i++) { y[i].re /= z0; y[i].im /= z0; }
}

static __thread const char *g_last_kernel = "";
extern "C" const char *qo_nodal_last_kernel(void) { return g_last_kernel; }
static __thread double g_last_compile_s = 0.0;
extern "C" double qo_nodal_last_compile_seconds(void) { return g_last_compile_s; }

/* ---- host: symbolic factorisation ------------------------------------------------------------------------- */
typedef std::vector<double2> cvec;

/* dense pivoted solve of one point on the host (reference for the static plan's self-check): returns the
 * solution columns X[j][i] for every port j and the row order the pivoting chose */
static bool host_dense(const NodalProg *hp, const double (*par)[4], double f, const double2 *yk, size_t yk_stride, std::vector<int> *perm_out, std::vector<cvec> *X)
{
    const int n = hp->n_unk, LD = QO_NODAL_MAX_UNK;
    cvec A((size_t)LD * LD, make_double2(0.0, 0.0));
    DenseSink<QO_NODAL_MAX_UNK> S = { A.data() };
    nodal_stamp_all(hp, par, 6.283185307179586476925286766559 * f, yk, yk_stride, S);
    std::vector<int> perm(n);
    for (int i = 0; i < n; i++) perm[i] = i;
    for (int c = 0; c < n; c++) {
        int piv = c;
        double best = A[c * LD + c].x * A[c * LD + c].x + A[c * LD + c].y * A[c * LD + c].y;
        for (int r = c + 1; r < n; r++) { const double2 v = A[r * LD + c]; const double m = v.x * v.x + v.y * v.y; if (m > best) { best = m; piv = r; } }
        if (!(best > 0.0)) return false;
        if (piv != c) { for (int j = 0; j < n; j++) std::swap(A[c * LD + j], A[piv * LD + j]); std::swap(perm[c], perm[piv]); }
        const double2 inv = hd_inv(A[c * LD + c]);
        for (int r = c + 1; r < n; r++) {
            const double2 l = hd_mul(A[r * LD + c], inv);
            A[r * LD + c] = l;
            for (int j = c + 1; j < n; j++) A[r * LD + j] = hd_fms(A[r * LD + j], l, A[c * LD + j]);
        }
    }
    if (perm_out) *perm_out = perm;
    if (X) {
        X->assign(hp->np, cvec(n));
        for (int j = 0; j < hp->np; j++) {
            cvec &x = (*X)[j];
            for (int i = 0; i < n; i++) x[i] = make_double2(perm[i] == hp->port_node[j] - 1 ? 1.0 / hp->port_z0[j] : 0.0, 0.0);
            for (int i = 1; i < n; i++) for (int q = 0; q < i; q++) x[i] = hd_fms(x[i], A[i * LD + q], x[q]);
            for (int i = n - 1; i >= 0; i--) { for (int q = i + 1; q < n; q++) x[i] = hd_fms(x[i], A[i * LD + q], x[q]); x[i] = hd_mul(x[i], hd_inv(A[i * LD + i])); }
        }
    }
    return true;
}

/* structural pattern of the stamps: a sink that only marks */
struct MarkSink {
    unsigned char *m;
    void add(int r, int c, double2) { m[r * QO_NODAL_MAX_UNK + c] = 1; }
};

/* Build the static plan; verify it at several grid points.  Returns false when the job should use the dense
 * kernel.  Unknowns are re-ordered so that the port nodes come LAST and, while the internal unknowns are being
 * eliminated, pivots are taken from the internal equations whenever one is close to the column maximum
 * (nodal matrices: the node's own KCL row; threshold 10 % of the column maximum).  The elimination then leaves the port block as the trailing Schur
 * complement, a port's unit right-hand side enters in the last rows, and the pruned substitutions touch only
 * that small trailing block instead of the whole factorisation. */
static bool build_static_thr(const NodalProg *hp, const double *f, int nf, const double2 *yb, NodalStatic *sp, double prefer_thr2);
static bool build_static(const NodalProg *hp, const double *f, int nf, const double2 *yb, NodalStatic *sp)
{
    /* internal-equation pivots preferred when within 10 % of the column maximum; if that order fails the
     * self-check (stiff networks at the band edge), plain partial pivoting at the reference point */
    return build_static_thr(hp, f, nf, yb, sp, 1e-2) || build_static_thr(hp, f, nf, yb, sp, 2.0);
}

static bool build_static_thr(const NodalProg *hp, const double *f, int nf, const double2 *yb, NodalStatic *sp, double prefer_thr2)
{
    const int n = hp->n_unk, np = hp->np, LD = QO_NODAL_MAX_UNK;
    memset(sp, 0, sizeof *sp);
    sp->n = n;
    /* column order: internal unknowns, then the port nodes in port order */
    std::vector<int> is_port(n, 0);
    for (int p = 0; p < np; p++) { if (is_port[hp->port_node[p] - 1]) return false; is_port[hp->port_node[p] - 1] = 1; }
    /* internal unknowns in greedy MINIMUM-DEGREE order on the structurally symmetrised pattern (eliminating an unknown joins
     * its neighbours): the bias networks are stars around their supply rails, and taking the leaves first leaves almost no
     * fill -- 175 -> 60 multiply-subtracts per point on the reference network against the netlist's own numbering. */
    int nc = 0;
    {
        std::vector<unsigned char> raw0((size_t)LD * LD, 0);
        MarkSink M0 = { raw0.data() };
        nodal_stamp_all(hp, hp->nom, 1.0, yb, (size_t)nf * 4, M0);
        std::vector<unsigned int> adj(n, 0);
        for (int r = 0; r < n; r++) for (int c = 0; c < n; c++) if (r != c && (raw0[r * LD + c] || raw0[c * LD + r])) adj[r] |= 1u << c;
        std::vector<int> gone(n, 0), comp(n, -1);
        /* unconnected sub-circuits (the reference network is two bias tees side by side) one after the other: the values of a
         * finished sub-circuit are dead before the next one is stamped, which halves the live set of the compiled kernel */
        int ncomp = 0;
        for (int u = 0; u < n; u++) {
            if (comp[u] >= 0) continue;
            std::vector<int> stack(1, u);
            comp[u] = ncomp;
            while (!stack.empty()) {
                const int a = stack.back();
                stack.pop_back();
                for (int v = 0; v < n; v++) if (((adj[a] >> v) & 1u) && comp[v] < 0) { comp[v] = ncomp; stack.push_back(v); }
            }
            ncomp++;
        }
        for (int step = 0; step < n - np; step++) {
            int best = -1, bdeg = 1 << 30, bcomp = 1 << 30;
            for (int u = 0; u < n; u++) {
                if (gone[u] || is_port[u]) continue;
                const int deg = __builtin_popcount(adj[u]);
                const int cu = comp[u];
                if (cu < bcomp || (cu == bcomp && deg < bdeg)) { bcomp = cu; bdeg = deg; best = u; }
            }
            gone[best] = 1;
            sp->colmap[best] = (uint8_t)nc++;
            const unsigned int nb_ = adj[best];
            for (int v = 0; v < n; v++) if ((nb_ >> v) & 1u) { adj[v] |= nb_; adj[v] &= ~(1u << v); adj[v] &= ~(1u << best); }
        }
    }
    for (int p = 0; p < np; p++) sp->colmap[hp->port_node[p] - 1] = (uint8_t)nc++;
    /* row (pivot) order from a numeric LU at a representative point, columns already permuted */
    const int k_ref = nf / 2;
    cvec D((size_t)LD * LD, make_double2(0.0, 0.0)), A((size_t)LD * LD, make_double2(0.0, 0.0));
    DenseSink<QO_NODAL_MAX_UNK> DS = { D.data() };
    nodal_stamp_all(hp, hp->nom, 6.283185307179586476925286766559 * f[k_ref], yb + (size_t)k_ref * 4, (size_t)nf * 4, DS);
    for (int r = 0; r < n; r++) for (int c = 0; c < n; c++) A[r * LD + sp->colmap[c]] = D[r * LD + c];
    std::vector<int> perm(n);
    for (int i = 0; i < n; i++) perm[i] = i;
    for (int c = 0; c < n; c++) {
        int piv = -1, piv_int = -1;
        double best = 0.0, best_int = 0.0;
        for (int r = c; r < n; r++) {
            const double2 v = A[r * LD + c];
            const double m = v.x * v.x + v.y * v.y;
            if (m > best) { best = m; piv = r; }
            if (!is_port[perm[r]] && m > best_int) { best_int = m; piv_int = r; }     /* rows 0..n_nodes-1 are node KCL equations */
        }
        if (piv < 0 || !(best > 0.0)) return false;
        if (c < n - np && piv_int >= 0 && best_int >= prefer_thr2 * best) piv = piv_int;     /* magnitudes squared */
        if (piv != c) { for (int j = 0; j < n; j++) std::swap(A[c * LD + j], A[piv * LD + j]); std::swap(perm[c], perm[piv]); }
        const double2 inv = hd_inv(A[c * LD + c]);
        for (int r = c + 1; r < n; r++) {
            const double2 l = hd_mul(A[r * LD + c], inv);
            if (l.x == 0.0 && l.y == 0.0) continue;
            A[r * LD + c] = l;
            for (int j = c + 1; j < n; j++) A[r * LD + j] = hd_fms(A[r * LD + j], l, A[c * LD + j]);
        }
    }
    for (int i = 0; i < n; i++) sp->rowmap[perm[i]] = (uint8_t)i;          /* equation perm[i] sits at pivot position i */
    /* structural pattern in (pivot row, permuted column) order, then symbolic elimination (fill) */
    std::vector<unsigned char> raw((size_t)LD * LD, 0), pat((size_t)LD * LD, 0);
    MarkSink M = { raw.data() };
    nodal_stamp_all(hp, hp->nom, 1.0, yb, (size_t)nf * 4, M);
    for (int r = 0; r < n; r++) for (int c = 0; c < n; c++) if (raw[r * LD + c]) pat[sp->rowmap[r] * LD + sp->colmap[c]] = 1;
    for (int c = 0; c < n; c++) {
        if (!pat[c * LD + c]) return false;                                 /* structurally zero pivot */
        for (int r = c + 1; r < n; r++)
            if (pat[r * LD + c])
                for (int j = c + 1; j < n; j++) if (pat[c * LD + j]) pat[r * LD + j] = 1;
    }
    int nnz = 0;
    for (int i = 0; i < LD * LD; i++) sp->pos[i] = -1;
    for (int r = 0; r < n; r++) for (int c = 0; c < n; c++) if (pat[r * LD + c]) sp->pos[r * LD + c] = (int16_t)nnz++;
    if (nnz > QN_NNZ_MAX) return false;
    sp->nnz = nnz;
    /* elimination program */
    std::vector<uint16_t> pg;
    auto P = [&](int r, int c) { return (uint16_t)sp->pos[r * LD + c]; };
    for (int c = 0; c < n; c++) {
        pg.push_back(P(c, c));
        std::vector<int> ucols, rows;
        for (int j = c + 1; j < n; j++) if (pat[c * LD + j]) ucols.push_back(j);
        for (int r = c + 1; r < n; r++) if (pat[r * LD + c]) rows.push_back(r);
        pg.push_back((uint16_t)ucols.size());
        for (int j : ucols) pg.push_back(P(c, j));
        pg.push_back((uint16_t)rows.size());
        for (int r : rows) { pg.push_back(P(r, c)); for (int j : ucols) pg.push_back(P(r, j)); }
    }
    /* per-port pruned substitution programs */
    std::vector<int> need(n, 0);
    for (int p = 0; p < np; p++) need[sp->colmap[hp->port_node[p] - 1]] = 1;
    for (int i = 0; i < n; i++)                     /* closure: a needed row needs every later unknown it references */
        if (need[i]) for (int q = i + 1; q < n; q++) if (pat[i * LD + q]) need[q] = 1;
    for (int j = 0; j < np; j++) {
        sp->solve_at[j] = (int32_t)pg.size();
        const int srow = sp->rowmap[hp->port_node[j] - 1];
        std::vector<int> reach(n, 0);
        reach[srow] = 1;
        std::vector<std::vector<int>> fterms(n);
        std::vector<int> frows;
        for (int i = srow + 1; i < n; i++) {
            for (int q = srow; q < i; q++) if (reach[q] && pat[i * LD + q]) fterms[i].push_back(q);
            if (!fterms[i].empty()) { reach[i] = 1; frows.push_back(i); }
        }
        pg.push_back((uint16_t)frows.size());
        for (int i : frows) { pg.push_back((uint16_t)i); pg.push_back((uint16_t)fterms[i].size()); for (int q : fterms[i]) { pg.push_back((uint16_t)q); pg.push_back(P(i, q)); } }
        std::vector<int> brows;
        for (int i = n - 1; i >= 0; i--) if (need[i]) brows.push_back(i);
        pg.push_back((uint16_t)brows.size());
        for (int i : brows) {
            std::vector<int> q;
            for (int c = i + 1; c < n; c++) if (pat[i * LD + c]) q.push_back(c);
            pg.push_back((uint16_t)i); pg.push_back(P(i, i)); pg.push_back((uint16_t)q.size());
            for (int c : q) { pg.push_back((uint16_t)c); pg.push_back(P(i, c)); }
        }
    }
    /* stamp stream: value index of every add() call in call order, first touches flagged; then the fill-only indices */
    {
        struct RecordSink {
            std::vector<uint16_t> *out; const NodalStatic *sp; std::vector<char> *touched;
            void add(int r, int c, double2) {
                const int q = sp->pos[sp->rowmap[r] * QO_NODAL_MAX_UNK + sp->colmap[c]];
                out->push_back((uint16_t)(q | ((*touched)[q] ? 0 : 0x8000)));
                (*touched)[q] = 1;
            }
        };
        std::vector<char> touched((size_t)nnz, 0);
        sp->stamp_at = (int32_t)pg.size();
        RecordSink RS = { &pg, sp, &touched };
        nodal_stamp_all(hp, hp->nom, 1.0, yb, (size_t)nf * 4, RS);
        sp->zero_at = (int32_t)pg.size();
        for (int q = 0; q < nnz; q++) if (!touched[q]) pg.push_back((uint16_t)q);
        sp->n_zero = (int32_t)pg.size() - sp->zero_at;
    }
    if (pg.size() > QN_PROG_MAX) return false;
    sp->prog_len = (int32_t)pg.size();
    memcpy(sp->prog, pg.data(), pg.size() * sizeof(uint16_t));
    /* self-check: the static program against the pivoted dense solve -- the nominal network at up to 33 grid points across the
     * band, then 8 pseudo-random vertices of the tolerance box (every random variable at +-1, a fixed Philox stream) at 9 grid
     * points each: a fixed pivot order that only suits the nominal values, or only part of the band, is rejected here; what
     * slips through (an interior sample at an unprobed frequency) is caught on the device by the multiplier guard (QN_GROWTH2) */
    const int n_nom = nf < 33 ? nf : 33, n_vert = hp->n_var > 0 ? 8 : 0, n_vp = nf < 9 ? nf : 9;
    double worst_l2 = 0.0;
    for (int t = 0; t < n_nom + n_vert * n_vp; t++) {
        const int vert = t < n_nom ? -1 : (t - n_nom) / n_vp;
        const int k = t < n_nom ? (n_nom > 1 ? (int)((long long)t * (nf - 1) / (n_nom - 1)) : 0)
                                : (n_vp > 1 ? (int)((long long)((t - n_nom) % n_vp) * (nf - 1) / (n_vp - 1)) : 0);
        double par[QO_NODAL_MAX_BR][4];
        for (int b = 0; b < hp->nb; b++)
            for (int q = 0; q < 4; q++) {
                double v = hp->nom[b][q];
                const int tv = hp->tvar[b][q];
                if (vert >= 0 && tv >= 0) {
                    const double x = qo_stream_variate(0x6e6f64616c706c6eull, (uint64_t)vert, (uint32_t)tv, 0) < 0.0 ? -1.0 : 1.0;
                    v = qo_stream_apply(v, hp->ttol[b][q], x, hp->tmode[b][q]);
                }
                par[b][q] = v;
            }
        std::vector<cvec> X;
        if (!host_dense(hp, par, f[k], yb + (size_t)k * 4, (size_t)nf * 4, NULL, &X)) return false;
        cvec V((size_t)nnz, make_double2(nan(""), nan("")));            /* poisoned: the streams must initialise every value */
        for (int i = 0; i < sp->n_zero; i++) V[sp->prog[sp->zero_at + i]] = make_double2(0.0, 0.0);
        ReplaySink S = { V.data(), sp->prog + sp->stamp_at, 0 };
        nodal_stamp_all(hp, par, 6.283185307179586476925286766559 * f[k], yb + (size_t)k * 4, (size_t)nf * 4, S);
        const double l2 = static_factor(sp->prog, n, V.data());
        if (getenv("QO100NET_NODAL_DEBUG") && !(l2 <= QN_GROWTH2)) fprintf(stderr, "qo_nodal: probe f=%g Hz: largest multiplier %.3g\n", f[k], sqrt(l2));
        if (!(l2 <= QN_GROWTH2)) return false;                          /* the device would flag this point: do not start on this plan */
        if (l2 > worst_l2) worst_l2 = l2;
        for (int j = 0; j < np; j++) {
            cvec x(n, make_double2(0.0, 0.0));
            x[sp->rowmap[hp->port_node[j] - 1]] = make_double2(1.0 / hp->port_z0[j], 0.0);
            static_solve(sp->prog, sp->solve_at[j], V.data(), x.data());
            for (int p = 0; p < np; p++) {
                const double2 a = x[sp->colmap[hp->port_node[p] - 1]], b = X[j][hp->port_node[p] - 1];
                const double err = hypot(a.x - b.x, a.y - b.y), ref = hypot(b.x, b.y);
                /* port voltages are O(1) (1/Z0 injected into ~Z0).  Entries that are exactly zero under per-point
                 * pivoting (reverse isolation of an ideal buffer) come out as ~1e-11 residues when the stiff
                 * reference network (100 uF next to 1.2 pF) is eliminated in the fixed ports-last order; 5e-11 on V
                 * = 1e-10 on S keeps the plan inside the 1e-9 parity bar, anything worse takes the dense kernel */
                if (!(err <= 1e-9 * ref + 5e-11)) {                                    /* NaN fails too */
                    if (getenv("QO100NET_NODAL_DEBUG")) fprintf(stderr, "qo_nodal: static plan rejected at f=%g Hz (%s), port %d<-%d: err %.3e ref %.3e\n", f[k], vert < 0 ? "nominal" : "tolerance-box vertex", p, j, err, ref);
                    return false;
                }
            }
        }
    }
    sp->worst_l2 = worst_l2;
    if (getenv("QO100NET_NODAL_DEBUG")) fprintf(stderr, "qo_nodal: static plan n=%d nnz=%d program=%d words, largest multiplier %.3g\n", n, nnz, sp->prog_len, sqrt(worst_l2));
    return true;
}

/* resident blocks per SM the compiled kernel is built for (64 threads each): 6 -> 168 registers */
#define QN_JIT_MINB 6
#include "qo_nodal_jit.h"

/* host-only front end: netlist + specs + tolerances -> device program, spec masks, block admittances */
static int nodal_compile(const qo_nodal *nd, const double *f, int nf, const qo_nspec *spec, int nspec, const qo_mc_cfg *cfg, int full,
                         NodalProg *hp, std::vector<unsigned char> &mask, std::vector<double2> &yb)
{
    if (!nd || !f || nf <= 0 || !cfg || nspec < 0 || nspec > QN_MAX_SPEC || (nspec && !spec)) { qo_set_error("bad arguments"); return QO_ERR_ARG; }
    if (nd->np < 1) { qo_set_error("the netlist has no ports"); return QO_ERR_ARG; }
    for (int k = 0; k < nf; k++) if (!(f[k] > 0.0) || !isfinite(f[k])) { qo_set_error("frequency %d is not a positive finite number", k); return QO_ERR_ARG; }
    memset(hp, 0, sizeof *hp);
    hp->n_nodes = nd->n_nodes; hp->nb = nd->nb; hp->np = nd->np; hp->full = full;
    hp->seed = cfg->seed; hp->dist = cfg->dist;
    if (hp->dist != QO_DIST_UNIFORM && hp->dist != QO_DIST_GAUSS3S) { qo_set_error("unknown distribution %d", hp->dist); return QO_ERR_ARG; }
    int n_unk = nd->n_nodes, n_sb = 0;
    for (int b = 0; b < nd->nb; b++) {
        hp->kind[b] = nd->br[b].kind;
        for (int k = 0; k < 4; k++) { hp->node[b][k] = nd->br[b].node[k]; hp->nom[b][k] = nd->br[b].p[k]; hp->tvar[b][k] = -1; }
        if (nd->br[b].kind == QO_NB_VCVS) n_unk++;
        if (nd->br[b].kind == QO_NB_SBLOCK) n_sb++;
    }
    if (n_unk > QO_NODAL_MAX_UNK) { qo_set_error("%d unknowns, limit %d", n_unk, QO_NODAL_MAX_UNK); return QO_ERR_RANGE; }
    hp->n_unk = n_unk;
    for (int p = 0; p < nd->np; p++) { hp->port_node[p] = nd->port_node[p]; hp->port_z0[p] = nd->port_z0[p]; }
    int nvar = 0;
    if (cfg->n_tol < 0 || (cfg->n_tol > 0 && !cfg->tol)) return QO_ERR_ARG;
    for (int i = 0; i < cfg->n_tol; i++) {
        const qo_tol *t = &cfg->tol[i];
        if (t->elem < 0 || t->elem >= nd->nb || t->param < 0 || t->param >= 4) { qo_set_error("tolerance %d: branch/param out of range", i); return QO_ERR_ARG; }
        if (t->var < 0 || t->var >= QN_MAX_VAR) { qo_set_error("tolerance %d: random variable index must be in [0,%d)", i, QN_MAX_VAR); return QO_ERR_RANGE; }
        if (nd->br[t->elem].kind == QO_NB_SBLOCK) { qo_set_error("tolerance %d: measured blocks carry no tolerances", i); return QO_ERR_ARG; }
        hp->tvar[t->elem][t->param] = (int16_t)t->var; hp->ttol[t->elem][t->param] = t->tol; hp->tmode[t->elem][t->param] = (uint8_t)(t->mode == QO_TOL_ABS);
        if (t->var + 1 > nvar) nvar = t->var + 1;
    }
    hp->n_var = nvar;
    hp->nspec = nspec;
    mask.assign((size_t)nf, 0);
    for (int s = 0; s < nspec; s++) {
        if (spec[s].kind != QO_SPEC_S21_MIN_DB && spec[s].kind != QO_SPEC_S21_MAX_DB) { qo_set_error("nodal spec %d: kind must be QO_SPEC_S21_MIN_DB or QO_SPEC_S21_MAX_DB", s); return QO_ERR_ARG; }
        if (spec[s].row < 0 || spec[s].row >= nd->np || spec[s].col < 0 || spec[s].col >= nd->np) { qo_set_error("nodal spec %d: S entry out of range", s); return QO_ERR_ARG; }
        hp->spec_min[s] = spec[s].kind == QO_SPEC_S21_MIN_DB; hp->spec_row[s] = spec[s].row; hp->spec_col[s] = spec[s].col;
        hp->spec_thr[s] = pow(10.0, spec[s].limit / 10.0); hp->spec_limit_db[s] = spec[s].limit;
        for (int k = 0; k < nf; k++) if (f[k] >= spec[s].f_lo && f[k] <= spec[s].f_hi) mask[k] |= (unsigned char)(1u << s);
    }
    hp->hist_bins = 0; hp->hist_spec = -1;
    if (!full && cfg->hist_bins > 0) {
        if (cfg->hist_bins > 1024 || cfg->hist_spec < 0 || cfg->hist_spec >= nspec || !(cfg->hist_hi > cfg->hist_lo)) { qo_set_error("bad histogram configuration"); return QO_ERR_ARG; }
        hp->hist_bins = cfg->hist_bins; hp->hist_spec = cfg->hist_spec; hp->hist_lo = cfg->hist_lo; hp->hist_hi = cfg->hist_hi;
    }
    /* measured blocks: admittance per (block branch, grid point), in branch order */
    yb.assign((size_t)n_sb * nf * 4, make_double2(0.0, 0.0));
    int ib = 0;
    for (int b = 0; b < nd->nb; b++) {
        if (nd->br[b].kind != QO_NB_SBLOCK) continue;
        const qo_s2p *blk = nd->blk[(int)nd->br[b].p[0]];
        for (int k = 0; k < nf; k++) {
            qo_c64 sv[4], y[4];
            qo_s2p_eval(blk, f[k], nd->br[b].p[1] != 0.0, sv);
            s_to_y(sv, nd->br[b].p[2], y);
            for (int q = 0; q < 4; q++) yb[((size_t)ib * nf + k) * 4 + q] = make_double2(y[q].re, y[q].im);
        }
        ib++;
    }
    return QO_OK;
}

/* what the host prepares for a nodal job */
struct NodalJob {
    NodalProg prog;
    NodalStatic plan;                   /* all zero unless use_static */
    bool use_static;                    /* the static plan was tried and passed its self-check */
    std::vector<unsigned char> mask;    /* per grid point: the specs that cover it (bit s) */
    std::vector<double2> yb;            /* measured blocks' admittances [block][nf][4]; one zero entry when there is none */
};

/* the host front end of every nodal entry point (needs no GPU): compile the netlist and, if try_static, the static plan */
static int nodal_prepare(const qo_nodal *nd, const double *f, int nf, const qo_nspec *spec, int nspec, const qo_mc_cfg *cfg, int full,
                         bool try_static, std::unique_ptr<NodalJob> &job)
{
    job.reset(new NodalJob());
    const int rc = nodal_compile(nd, f, nf, spec, nspec, cfg, full, &job->prog, job->mask, job->yb);
    if (rc) return rc;
    if (job->yb.empty()) job->yb.assign(4, make_double2(0.0, 0.0));
    job->use_static = try_static && build_static(&job->prog, f, nf, job->yb.data(), &job->plan);
    return QO_OK;
}

/* The host-only part of a nodal job (needs no GPU): compile the netlist and try the static (symbolic) factorisation plan.
 * info[0] = static plan accepted (0/1), [1] = unknowns, [2] = packed non-zeros incl. fill, [3] = program length (16-bit words);
 * *max_multiplier = largest |L| entry the plan-time probes met (per-point partial pivoting would keep it <= 1). */
extern "C" int qo_nodal_analyze(const qo_nodal *nd, const double *f, int nf, const qo_mc_cfg *cfg, int info[4], double *max_multiplier)
{
    qo_clear_error();
    if (!info) return QO_ERR_ARG;
    QoNodalOverrides ov;                     /* the analysis tries the static plan whatever they say, but a bad value is refused */
    int rc = qo_nodal_overrides_read(&ov);
    if (rc) return rc;
    qo_mc_cfg c0;
    memset(&c0, 0, sizeof c0);
    std::unique_ptr<NodalJob> job;
    rc = nodal_prepare(nd, f, nf, NULL, 0, cfg ? cfg : &c0, 1, true, job);
    if (rc) return rc;
    const bool ok = job->use_static;
    info[0] = ok; info[1] = job->prog.n_unk; info[2] = ok ? job->plan.nnz : 0; info[3] = ok ? job->plan.prog_len : 0;
    if (max_multiplier) *max_multiplier = ok ? sqrt(job->plan.worst_l2) : 0.0;
    return QO_OK;
}

/* Host-only as well (NVRTC compiles without a GPU): print the static plan of this job as a kernel, compile it for sm_100a and
 * report what ptxas made of it.  info[0] = compiled (0/1; 0 also when the static plan is refused or libnvrtc is missing),
 * [1] = registers per thread, [2] = stack frame bytes (0 = every value of the factorisation lives in registers), [3] = spill
 * bytes, [4] = complex multiply-subtracts per point, [5] = reciprocals per point. */
extern "C" int qo_nodal_jit_analyze(const qo_nodal *nd, const double *f, int nf, const qo_nspec *spec, int nspec, const qo_mc_cfg *cfg, int info[6])
{
    qo_clear_error();
    if (!info || !cfg) return QO_ERR_ARG;
    for (int i = 0; i < 6; i++) info[i] = 0;
    QoNodalOverrides ov;                     /* as in qo_nodal_analyze: read only to refuse a bad value */
    int rc = qo_nodal_overrides_read(&ov);
    if (rc) return rc;
    std::unique_ptr<NodalJob> job;
    rc = nodal_prepare(nd, f, nf, spec, nspec, cfg, cfg->mode == QO_MODE_FULL_S, true, job);
    if (rc) return rc;
    if (!job->use_static) { qo_set_error("the static plan failed its self-check for this network"); return QO_OK; }
    const QnJitEntry *e = qn_jit_get(&job->prog, &job->plan, false, true);
    info[0] = e->ok; info[1] = e->regs; info[2] = e->stack_bytes; info[3] = e->spill_bytes; info[4] = e->n_fms; info[5] = e->n_inv;
    if (!e->ok) qo_set_error("%s", e->log.substr(0, 400).c_str());
    return QO_OK;
}

/* points below which a job is not worth a compilation (0.3 - 1 s of NVRTC against 8e8 points/s on the interpreted kernel); a
 * kernel this process has already compiled is used from QN_JIT_MIN_CACHED points on */
#define QN_JIT_MIN_POINTS 400000000ull
#define QN_JIT_MIN_CACHED 1000000ull

/* the interpreted kernel of a job: the static plan's instantiation by its number of values, the dense one by its unknowns */
static const void *nodal_kernel(bool use_static, int nnz, int n_unk)
{
    if (use_static) {
        if (nnz <= 64) return (const void *)qo_nodal_kernel<32, 1, 64>;
        if (nnz <= 128) return (const void *)qo_nodal_kernel<32, 1, 128>;
        if (nnz <= 256) return (const void *)qo_nodal_kernel<32, 1, 256>;
        return (const void *)qo_nodal_kernel<32, 1, QN_NNZ_MAX>;
    }
    if (n_unk <= 8) return (const void *)qo_nodal_kernel<8, 0, 1>;
    if (n_unk <= 16) return (const void *)qo_nodal_kernel<16, 0, 1>;
    if (n_unk <= 24) return (const void *)qo_nodal_kernel<24, 0, 1>;
    return (const void *)qo_nodal_kernel<32, 0, 1>;
}

static int nodal_run(qo_ctx *ctx, const qo_nodal *nd, const double *f, int nf, const qo_nspec *spec, int nspec,
                     const qo_mc_cfg *cfg, qo_mc_result *res, qo_c64 *full_s_host)
{
    if (!ctx || !cfg) { qo_set_error("bad arguments"); return QO_ERR_ARG; }
    g_last_compile_s = 0.0;
    const int full = cfg->mode == QO_MODE_FULL_S;
    if (full && !full_s_host) { qo_set_error("FULL_S needs an output buffer"); return QO_ERR_ARG; }
    if (!full && !res) return QO_ERR_ARG;
    QoNodalOverrides ov;
    int rc = qo_nodal_overrides_read(&ov);
    if (rc) return rc;
    /* static (symbolic) plan unless forced off or its self-check fails */
    std::unique_ptr<NodalJob> job;
    rc = nodal_prepare(nd, f, nf, spec, nspec, cfg, full, ov.kernel != QoNodalOverrides::DENSE, job);
    if (rc) return rc;
    const NodalProg *hp = &job->prog;
    bool use_static = job->use_static;
    if (ov.kernel == QoNodalOverrides::STATIC && !use_static) { qo_set_error("QO100NET_NODAL=static: the static plan failed its self-check for this network"); return QO_ERR_UNSUPPORTED; }
    const int ncnt = 2 + nspec + hp->hist_bins;
    const unsigned long long N = cfg->n_samples;
    if (N == 0) { if (res) { res->n_pass = res->n_total = 0; } return QO_OK; }
    /* the plan compiled into a kernel of its own: large jobs (QO100NET_NODAL=jit: always; =static / =dense: never) */
    const QnJitEntry *jit = NULL;
    if (use_static && ov.kernel != QoNodalOverrides::STATIC) {
        const bool forced = ov.kernel == QoNodalOverrides::JIT;
        const unsigned long long npts = N * (unsigned long long)nf;
        if (forced || npts >= QN_JIT_MIN_CACHED) {
            const size_t had = g_qn_jit.size();
            jit = qn_jit_get(hp, &job->plan, true, forced || npts >= QN_JIT_MIN_POINTS);
            if (jit && g_qn_jit.size() != had) g_last_compile_s = jit->compile_s;
            if (jit && !jit->ok) {
                if (forced) { qo_set_error("QO100NET_NODAL=jit: %s", jit->log.substr(0, 400).c_str()); return QO_ERR_UNSUPPORTED; }
                jit = NULL;
            }
        }
    } else if (ov.kernel == QoNodalOverrides::JIT) { qo_set_error("QO100NET_NODAL=jit: the static plan failed its self-check for this network"); return QO_ERR_UNSUPPORTED; }
    const void *kern = jit ? (const void *)jit->kern : nodal_kernel(use_static, job->plan.nnz, hp->n_unk);

    /* samples are independent: GPU g of the ctx takes the contiguous range [N g / G, N (g+1) / G) of the job (the Philox counter
     * carries the global sample index, so the counters do not depend on G); the host adds the u64 counters, FULL_S slabs are
     * copied back one after the other */
    const int G = (N >= (unsigned long long)ctx->ndev * 64ull) ? ctx->ndev : 1;
    struct NodalDev {
        NodalProg *dprog; NodalStatic *dsp; double *dfr; unsigned char *dmask; double2 *dy, *ds; unsigned long long *dcnt;
        unsigned long long off, n;
        int grid;
    } nv[8];
    memset(nv, 0, sizeof nv);
    const int np_ = nd->np;
    std::vector<unsigned long long> h((size_t)ncnt + 1, 0ull), hg((size_t)ncnt + 1);
    float ms_max = 0.0f;
    int chunk_len = nf, nchunks = 1;
    /* FULL_S: cut the grid into QN_TPB-point chunks so that a nominal sweep fills the GPU */
    if (full) { chunk_len = QN_TPB; nchunks = (nf + chunk_len - 1) / chunk_len; }
    double growth2 = ov.growth2 > 0.0 ? ov.growth2 : QN_GROWTH2;
#define CUN(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { qo_set_error("%s -> %s", #call, cudaGetErrorString(e_)); rc = e_ == cudaErrorMemoryAllocation ? QO_ERR_NOMEM : QO_ERR_CUDA; goto out; } } while (0)
    for (int g = 0; g < G; g++) {
        DevCtx *dc = &ctx->d[g];
        NodalDev &v = nv[g];
        v.off = N * (unsigned long long)g / (unsigned long long)G;
        v.n = N * (unsigned long long)(g + 1) / (unsigned long long)G - v.off;
        CUN(cudaSetDevice(dc->device));
        CUN(cudaMallocAsync((void **)&v.dprog, sizeof(NodalProg), dc->stream));
        CUN(cudaMallocAsync((void **)&v.dsp, sizeof(NodalStatic), dc->stream));
        CUN(cudaMemcpyAsync(v.dsp, &job->plan, sizeof(NodalStatic), cudaMemcpyHostToDevice, dc->stream));
        CUN(cudaMallocAsync((void **)&v.dfr, (size_t)nf * sizeof(double), dc->stream));
        CUN(cudaMallocAsync((void **)&v.dmask, (size_t)nf, dc->stream));
        CUN(cudaMallocAsync((void **)&v.dy, job->yb.size() * sizeof(double2), dc->stream));
        CUN(cudaMallocAsync((void **)&v.dcnt, (size_t)(ncnt + 1) * sizeof(unsigned long long), dc->stream));     /* + the suspect-point counter of the static kernels */
        if (full) CUN(cudaMallocAsync((void **)&v.ds, (size_t)v.n * nf * np_ * np_ * sizeof(double2), dc->stream));
        CUN(cudaMemcpyAsync(v.dprog, hp, sizeof(NodalProg), cudaMemcpyHostToDevice, dc->stream));
        CUN(cudaMemcpyAsync(v.dfr, f, (size_t)nf * sizeof(double), cudaMemcpyHostToDevice, dc->stream));
        CUN(cudaMemcpyAsync(v.dmask, job->mask.data(), (size_t)nf, cudaMemcpyHostToDevice, dc->stream));
        CUN(cudaMemcpyAsync(v.dy, job->yb.data(), job->yb.size() * sizeof(double2), cudaMemcpyHostToDevice, dc->stream));
        /* persistent grid = exactly the resident blocks (a larger grid runs in 1.6 waves: 4.0e8 instead of 4.4e8
         * points/s on the reference network); latency hiding matters more here than the private arrays' L2 footprint */
        int bps = 0;
        if (jit) {
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, QN_TPB, 0) != cudaSuccess || bps <= 0) {
                cudaGetLastError();
                bps = jit->regs > 0 ? 65536 / (((jit->regs + 7) & ~7) * QN_TPB) : 4;
                if (bps > 16) bps = 16;
            }
        } else if (use_static) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, QN_TPB, 0);
        if (bps <= 0) bps = 8;
        const unsigned long long units = v.n * (unsigned long long)nchunks;
        const unsigned long long cap = (unsigned long long)dc->sm_count * (unsigned long long)bps;
        v.grid = (int)(units < cap ? units : cap);
    }
    /* some (sample, frequency) point met a multiplier above the guard (or a NaN) under the static plan's fixed pivot order: the
     * whole job is redone once with per-point partial pivoting, on the grid computed above */
    for (int attempt = 0; attempt < 2; attempt++) {
        g_last_kernel = jit ? "qo_nodal_jit_kernel" : use_static ? "qo_nodal_kernel<static,local>" : "qo_nodal_kernel<dense>";
        for (int g = 0; g < G; g++) {
            DevCtx *dc = &ctx->d[g];
            NodalDev &v = nv[g];
            unsigned long long off_g = cfg->sample_offset + v.off;
            void *args[] = { &v.dprog, &v.dsp, &v.dfr, &v.dmask, &v.dy, &nf, &chunk_len, &nchunks, &off_g, &v.n, &v.dcnt, &v.ds, &growth2 };
            void *args_jit[] = { &v.dprog, &v.dfr, &v.dmask, &v.dy, &nf, &chunk_len, &nchunks, &off_g, &v.n, &v.dcnt, &v.ds, &growth2 };   /* the plan is compiled in */
            CUN(cudaSetDevice(dc->device));
            CUN(cudaMemsetAsync(v.dcnt, 0, (size_t)(ncnt + 1) * sizeof(unsigned long long), dc->stream));
            cudaEventRecord(dc->ev0, dc->stream);
            CUN(cudaLaunchKernel(kern, dim3((unsigned)v.grid), dim3(QN_TPB), jit ? args_jit : args, 0, dc->stream));
            cudaEventRecord(dc->ev1, dc->stream);
            CUN(cudaGetLastError());
        }
        for (size_t i = 0; i < h.size(); i++) h[i] = 0ull;
        ms_max = 0.0f;
        for (int g = 0; g < G; g++) {
            DevCtx *dc = &ctx->d[g];
            CUN(cudaSetDevice(dc->device));
            CUN(cudaStreamSynchronize(dc->stream));
            CUN(cudaMemcpy(hg.data(), nv[g].dcnt, (size_t)(ncnt + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < h.size(); i++) h[i] += hg[i];
            float ms = 0;
            cudaEventElapsedTime(&ms, dc->ev0, dc->ev1);
            if (ms > ms_max) ms_max = ms;
        }
        if (!use_static || h[ncnt] == 0) break;
        if (ov.kernel == QoNodalOverrides::STATIC) { qo_set_error("QO100NET_NODAL=static: %llu points needed another pivot order", h[ncnt]); rc = QO_ERR_UNSUPPORTED; goto out; }
        if (getenv("QO100NET_NODAL_DEBUG")) fprintf(stderr, "qo_nodal: %llu suspect points under the static plan, re-running on the dense kernel\n", h[ncnt]);
        use_static = false;
        jit = NULL;
        kern = nodal_kernel(false, 0, hp->n_unk);
    }
    if (full)
        for (int g = 0; g < G; g++) {
            CUN(cudaSetDevice(ctx->d[g].device));
            CUN(cudaMemcpy(full_s_host + (size_t)nv[g].off * nf * np_ * np_, nv[g].ds, (size_t)nv[g].n * nf * np_ * np_ * sizeof(double2), cudaMemcpyDeviceToHost));
        }
    if (res) {
        const int n_unk = hp->n_unk;
        res->n_pass = full ? 0 : h[0];
        res->n_total = full ? N : h[1];
        if (res->fail_per_spec) for (int s = 0; s < nspec; s++) res->fail_per_spec[s] = h[2 + s];
        if (res->hist) for (int b = 0; b < hp->hist_bins; b++) res->hist[b] = h[2 + nspec + b];
        res->seconds = ms_max * 1e-3;
        res->evals_per_s = ms_max > 0 ? (double)N * nf / (ms_max * 1e-3) : 0.0;
        res->flops_per_eval = (8.0 / 3.0) * n_unk * n_unk * n_unk + 8.0 * nd->np * n_unk * n_unk;   /* DENSE LU + substitutions, real flops */
    }
out:
#undef CUN
    for (int g = 0; g < G; g++) {
        void *ptrs[] = { nv[g].dprog, nv[g].dsp, nv[g].dfr, nv[g].dmask, nv[g].dy, nv[g].dcnt, nv[g].ds };
        cudaSetDevice(ctx->d[g].device);
        for (size_t i = 0; i < sizeof ptrs / sizeof ptrs[0]; i++) if (ptrs[i]) cudaFreeAsync(ptrs[i], ctx->d[g].stream);
    }
    cudaSetDevice(ctx->d[0].device);
    return rc;
}

extern "C" int qo_nodal_mc_run(qo_ctx *ctx, const qo_nodal *nd, const double *f, int nf, const qo_nspec *spec, int nspec,
                               const qo_mc_cfg *cfg, qo_mc_result *res, qo_c64 *full_s)
{
    qo_clear_error();
    return nodal_run(ctx, nd, f, nf, spec, nspec, cfg, res, full_s);
}

extern "C" int qo_nodal_sweep(qo_ctx *ctx, const qo_nodal *nd, const double *f, int nf, qo_c64 *s)
{
    qo_clear_error();
    if (!s) return QO_ERR_ARG;
    qo_mc_cfg cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.n_samples = 1; cfg.mode = QO_MODE_FULL_S; cfg.precision = 64;
    return nodal_run(ctx, nd, f, nf, NULL, 0, &cfg, NULL, s);
}
