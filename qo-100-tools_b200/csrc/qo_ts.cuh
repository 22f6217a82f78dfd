/*
 * qo_ts.cuh -- thread-per-sample flavour of the transfer-function Monte-Carlo kernel (sm_100a, FP64).
 *
 * Same job and same mathematics as qo_tf.cuh (reduce-only |S21| yield of the pcb/generic-filter ladder family, reference
 * pcb/generic-filter/README.md:13, qo-100-generic-filter.sch:1450-1488,1703-1995; behind the coupled-line block of
 * util/directional-couplers/dir_cpl_2.4g_20dB.trc:18-20 for BASELINE config 5): per sample the cascade is expanded into real
 * polynomials in s, per point they are evaluated by Horner in y = -x^2.  What changes is who holds the coefficients.
 *
 * In qo_mc_tf_kernel one WARP owns a sample: lanes own different frequencies and every Horner step re-reads the sample's
 * coefficients from shared memory -- one LDS.128 per 16 DFMA.  tools/horner_probe*.cu measured what that costs on a B200: a
 * Horner loop fed from shared memory peaks at 77-81 % of the FP64 pipe whatever the prefetch distance, the same loop with its
 * coefficients in registers at 90-92 %.  Registers can only hold the coefficients if a THREAD owns the sample, so here a
 * thread does everything for its sample, and nothing is shared:
 *
 *   stage A  variates (the same bit-exact Philox stream, one call per perturbed parameter), element records, and the
 *            expansion of [P; Q] and E as TRUNCATED polynomials in registers.  Multiplying by a branch's (a0 + a1 s + a2 s^2)
 *            only moves coefficients upwards, so the 2 KN lowest coefficients of P, Q and the KE lowest of E -- the ones the
 *            plan keeps -- are exact without ever forming the higher ones.  Register arrays need static indices: there is one
 *            kernel per numerator length KN, carrying one body per denominator length KE, up to the capacities below;
 *   stage C  the frequency loop runs over ALL grid points per thread, PT points in flight.  The grid value y is the same for
 *            the whole warp (a broadcast load per group of points, nothing per Horner step), every DFMA takes its coefficient
 *            from a register, the per-spec sign accumulators / the histogram tracker are thread-private: no shuffles, no
 *            shared memory, no warp reduction inside or after the loop.  The grid is walked as a few runs of groups that see
 *            the same spec bits, so the bookkeeping branches on loop-invariant warp-uniform predicates.  Where one |S21| spec
 *            alone looks (a stop band) only the sign of its margin N2 - t E matters, and that is one polynomial in y of
 *            max(2 KN, KE) coefficients: the plan accepts it per spec where it stays within 1e-12 of |den|^2 of the unfused
 *            margin (qo_tf.cu::tf_fuse_gate -- a stop band does, a ripple pass band usually not) and puts that spec's runs
 *            last; after the other runs the thread forms the polynomial once in double-double (qo_tf_core.h::qo_tf_fuse, in the
 *            registers of the expansion, which are dead by then) and walks the runs with one Horner chain per point:
 *            2 KN - 1 or KE - 1 DFMA per point instead of 2 (KN - 1) + (KE - 1) + 4 (cfg2: 17 instead of 33);
 *   stage D  verdict per thread, counters by warp ballots, the histogram value (a log10) at full lane efficiency.
 *
 * Stage A costs ~4 500 instructions per sample against ~180 000 for the loop (the warp-cooperative expansion of qo_tf.cuh:
 * ~1 600 WARP instructions per sample against ~5 800), so there is nothing left to overlap.  Warps take batches of 32 samples
 * from a ticket counter; the launcher hands the last n mod 32 samples of a launch to qo_mc_tf_kernel.
 * Jobs outside the capacities, |S11| / group-delay specs, more than four specs, the physical coupler element: qo_mc_tf_kernel.
 */
#pragma once
#include "qo_tf.cuh"

#define QO_TS_TPB 128
/* points in flight per thread / resident blocks per SM (both at 168 registers, 12 warps per SM): plain ladders hold <= 36
 * coefficients (72 registers) and run four points -- at 128 registers (4 blocks) ptxas serialises the four Horner chains and
 * the kernel is 8 % slower; behind a coupled-line block P and Q stay apart (<= 40 coefficients + the block's constants and the
 * rotating angle), two points */
#define QO_TS_PT2 4
#define QO_TS_MINB2 3
#define QO_TS_PT4 2
#define QO_TS_FG2 3              /* fused runs of plain ladders (one Horner chain per point): groups walked at once -- 12 points in flight;
                                    cfg2 on a B200 at its 1000 W limit: 4 points 4.97e11 evals/s, 8 points 5.32e11, 12 points 5.41e11, 16 points 5.40e11 */
#define QO_TS_MINB4 3
#define QO_TS_CAPN2 10           /* plain ladders (NN = 2): numerator coefficient pairs held in registers */
#define QO_TS_CAPE2 16           /* ... and E coefficients */
#define QO_TS_CAPN4 8            /* behind a coupled-line block (NN = 4: P and Q apart) */
#define QO_TS_CAPE4 8

#define QO_TS_MAXRUN 40          /* <= 4 band edges per spec, each at most one straddling group */
#define QO_PTS_N(n) _Pragma("unroll") for (int p = 0; p < (n); p++)

struct TsParams {
    TfParams t;                          /* the job, exactly as qo_mc_tf_kernel takes it */
    const double *y1, *x1;               /* per POINT: -(w/wref)^2 and w/wref (the same tables, read as scalars) */
    const uint2 *mw;                     /* per point: byte masks of specs 0-3 (x) and 4-7 (y) */
    struct { int g0, ngroups; unsigned int any, all; } runs[QO_TS_MAXRUN];  /* runs of groups (PT points each) that see the same spec bits */
    int nruns;
    int nplain;                          /* runs[0, nplain): walked on |numerator|^2 and E; runs[nplain, nruns): the runs of the one
                                            fused spec (walked on its margin polynomial, qo_tf_fuse) */
    int npt;                             /* points to walk: the grid rounded up to a whole group (padding carries no spec bit) */
    unsigned long long nbatches;         /* 32-sample batches, handed to the warps through a ticket counter */
    unsigned long long *ticket;          /* zeroed per launch */
    double w0, dw;                       /* coupler on a uniform grid: first angular frequency and step */
};

/* stage C for one (KN, KE): everything in registers.
 * The grid is walked as a few RUNS of groups (PT points each) that see the same spec bits (TsParams::runs, built by the
 * plan from the band edges): inside a run the spec bookkeeping branches on loop-invariant, warp-uniform predicates -- nothing
 * is loaded or decoded per group except the PT grid values themselves.  Groups that straddle a band edge are runs of their own
 * and take their per-point byte masks. */
template <int NN, int KN, int KE, bool CPL, int NS, int PT>
__device__ __forceinline__ void ts_loop(const TsParams &Q, unsigned long long sample, unsigned int (&acc)[NS], double &trkv)
{
    static_assert(PT == 2 || PT == 4, "two or four points in flight");
    constexpr int NC = 2 * KN;           /* kept coefficients per numerator polynomial */
    static_assert(KN >= 2 && (KE == 0 || KE >= 2), "the plan keeps at least two rows");
    const TfParams &P = Q.t;
    const DevProg *__restrict__ prog = P.prog;
    double cn[NN * KN], ce[KE > 0 ? KE : 1];
    {
        /* stage A: truncated expansion from the load end, same operation order per coefficient as tf_sample_stage */
        double pc[NC], qc[NC], ec[KE > 0 ? KE : 1];
#pragma unroll
        for (int i = 0; i < NC; i++) { pc[i] = 0.0; qc[i] = 0.0; }
#pragma unroll
        for (int i = 0; i < KE; i++) ec[i] = 0.0;
        pc[0] = P.rl; qc[0] = P.zn; ec[0] = 1.0;
        for (int e = P.n_el - 1; e >= 0; e--) {
            const int ge = P.el0 + e;
            double pr[6];
#pragma unroll
            for (int k = 0; k < 6; k++) {
                pr[k] = prog->nom[ge][k];
                const int tv = prog->tvar[ge][k];
                if (tv >= 0) pr[k] = qo_stream_apply(pr[k], prog->ttol[ge][k], qo_stream_variate(P.seed, P.sample_offset + sample, (uint32_t)tv, P.dist), prog->tmode[ge][k]);
            }
            double nd[6];
            const int series = qo_tf_element(prog->opcode[ge], pr, P.wref, nd);
            const double sc = series ? P.zni : P.zn;
            const double n0 = nd[0] * sc, n1 = nd[1] * sc, n2_ = nd[2] * sc, d0 = nd[3], d1 = nd[4], d2 = nd[5];
#pragma unroll
            for (int i = NC - 1; i >= 0; i--) {
                const double p0 = pc[i], p1 = i >= 1 ? pc[i - 1] : 0.0, p2 = i >= 2 ? pc[i - 2] : 0.0;
                const double q0 = qc[i], q1 = i >= 1 ? qc[i - 1] : 0.0, q2 = i >= 2 ? qc[i - 2] : 0.0;
                const double dp = fma(d0, p0, fma(d1, p1, d2 * p2)), dq = fma(d0, q0, fma(d1, q1, d2 * q2));
                if (series) { pc[i] = fma(n0, q0, fma(n1, q1, fma(n2_, q2, dp))); qc[i] = dq; }      /* Z = N/D: P <- D P + N Q, Q <- D Q */
                else { qc[i] = fma(n0, p0, fma(n1, p1, fma(n2_, p2, dq))); pc[i] = dp; }             /* Y = N/D: Q <- D Q + N P, P <- D P */
            }
            if (KE > 0) {
                const double e0 = d0 * d0, e1 = fma(2.0 * d0, d2, -d1 * d1), e2 = d2 * d2;          /* |D(jx)|^2 in y */
#pragma unroll
                for (int i = KE - 1; i >= 0; i--)
                    ec[i] = fma(e0, ec[i], fma(e1, i >= 1 ? ec[i - 1] : 0.0, e2 * (i >= 2 ? ec[i - 2] : 0.0)));
            }
        }
        const double zq0 = P.rs * P.zni;
#pragma unroll
        for (int k = 0; k < KN; k++) {
            if (NN == 4) { cn[k * 4] = pc[2 * k]; cn[k * 4 + 1] = pc[2 * k + 1]; cn[k * 4 + 2] = qc[2 * k]; cn[k * 4 + 3] = qc[2 * k + 1]; }
            else { cn[k * NN] = fma(zq0, qc[2 * k], pc[2 * k]); cn[k * NN + 1] = fma(zq0, qc[2 * k + 1], pc[2 * k + 1]); }
        }
#pragma unroll
        for (int k = 0; k < KE; k++) ce[k] = ec[k];
    }
    /* coupled-line block, equal mode angles on a uniform grid (qo_tf.cuh::tf_cpl_matched_same): five constants and the angle,
     * carried from point to point by one rotation */
    double k0x = 0, k0y = 0, k2x = 0, k2y = 0, k4 = 0, sn = 0, cs = 1, st_s = 0, st_c = 1;
    if (CPL) {
        double xv[QO_MAX_VAR], o[QO_LAD_CPL], nom_k[2];
        for (int v = 0; v < P.n_var; v++) xv[v] = qo_stream_variate(P.seed, P.sample_offset + sample, (uint32_t)v, P.dist);
        lad_derive<double>(prog, P.cpl_op, xv, o, NULL, nom_k);
        const double cE = o[0], hE = o[1], cO = o[2], hO = o[3];
        const double k1 = cE * cO, k2 = cE + cO, k3 = fma(hE, cO, hO * cE), k4_ = hE + hO;
        k0x = k1 - k3; k0y = k1 + k3; k2x = 2.0 * (k2 - k4_); k2y = 2.0 * (k2 + k4_); k4 = k2 * k2;
        sincos(o[4] * Q.w0, &sn, &cs);
        sincos(o[4] * Q.dw, &st_s, &st_c);
    }
    const int hs = P.hist_spec;
    const bool hneg = hs >= 0 && P.neg[hs & (QO_TF_NSPEC - 1)];
    const double zq = P.rs * P.zni;
    double y[PT];
#pragma unroll
    for (int h = 0; h < PT; h += 2) { const double2 a = __ldg((const double2 *)(Q.y1 + h)); y[h] = a.x; y[h + 1] = a.y; }
    /* one group of PT points: all NN * PT numerator chains and the PT chains of E advance together (one long stream of
     * independent FMAs), then |numerator|^2 (behind a coupler: contracted with the block's row vector), and -- y being dead by
     * then -- the request for the next group's grid values (the tables carry padding beyond the grid).
     * Leaves n2[PT], dd[PT]:  |den|^2 = n2 / dd. */
#define QO_TS_CORE                                                                                                   \
        const int j = gi * PT;                                                                                       \
        double r[NN][PT], dd[PT], n2[PT];                                                                            \
        _Pragma("unroll") for (int c = 0; c < NN; c++) { QO_PTS_N(PT) r[c][p] = fma(cn[NN * (KN - 1) + c], y[p], cn[NN * (KN - 2) + c]); } \
        if (KE >= 2) { QO_PTS_N(PT) dd[p] = fma(ce[KE - 1], y[p], ce[KE - 2]); }                                     \
        else { QO_PTS_N(PT) dd[p] = 1.0; }                                                                           \
        _Pragma("unroll") for (int s_ = 0; s_ < (KN - 2 > KE - 2 ? KN - 2 : KE - 2); s_++) {                         \
            if (s_ < KN - 2) {                                                                                       \
                _Pragma("unroll") for (int c = 0; c < NN; c++) { QO_PTS_N(PT) r[c][p] = fma(r[c][p], y[p], cn[NN * (KN - 3 - s_) + c]); } \
            }                                                                                                        \
            if (s_ < KE - 2) { QO_PTS_N(PT) dd[p] = fma(dd[p], y[p], ce[KE - 3 - s_]); }                             \
        }                                                                                                            \
        if (!CPL) {                                                                                                  \
            QO_PTS_N(PT) { const double t_ = r[1][p] * r[1][p]; n2[p] = fma(-y[p], t_, r[0][p] * r[0][p]); }         \
        } else {                                                                                                     \
            double x[PT];                                                                                            \
            _Pragma("unroll") for (int h = 0; h < PT; h += 2) { const double2 a_ = __ldg((const double2 *)(Q.x1 + j + h)); x[h] = a_.x; x[h + 1] = a_.y; } \
            QO_PTS_N(PT) {                                                                                           \
                const double c2 = cs * cs, s2 = sn * sn, sc = cs * sn, c4 = 4.0 * c2;                                \
                const double uar = fma(-k0x, s2, c4), ubr = fma(-k0y, s2, c4), uai = k2x * sc, ubi = k2y * sc;       \
                const double sg2 = fma(k4, s2, 4.0 * c4);                                                            \
                const double pi_ = r[1][p] * x[p], qr = r[NN - 2][p] * zq, qi = (r[NN - 1][p] * x[p]) * zq;          \
                const double nr = fma(uar, r[0][p], fma(-uai, pi_, fma(ubr, qr, -ubi * qi)));                        \
                const double ni = fma(uar, pi_, fma(uai, r[0][p], fma(ubr, qi, ubi * qr)));                          \
                n2[p] = fma(nr, nr, ni * ni);                                                                        \
                dd[p] *= sg2;                                                                                        \
                const double s1 = fma(sn, st_c, cs * st_s), c1 = fma(cs, st_c, -sn * st_s);                          \
                sn = s1; cs = c1;                                                                                    \
            }                                                                                                        \
        }                                                                                                            \
        _Pragma("unroll") for (int h = 0; h < PT; h += 2) { const double2 a_ = __ldg((const double2 *)(Q.y1 + j + PT + h)); y[h] = a_.x; y[h + 1] = a_.y; }
#define QO_TS_VALUE                                                                                                  \
        double val[PT];                                                                                              \
        if (KE < 2 && !CPL) { QO_PTS_N(PT) val[p] = n2[p]; }                                                         \
        else { double rd[PT]; lad_rcp_batch<PT>(dd, rd); QO_PTS_N(PT) val[p] = fabs(n2[p] * rd[p]); }   /* |.|: see qo_tf.cuh */
    /* spec bookkeeping as in qo_mc_tf_kernel: the histogram spec tracks the value n2 / dd, every other spec the sign of
     * thr dd - n2 (or n2 - thr dd).  Inside a run the active specs do not change, so the common cases -- exactly one spec
     * active, or none -- get loops of their own with nothing to decide per group. */
    unsigned int idle = 0u;              /* points that no spec looks at are evaluated all the same (the metric counts them) and land in
                                            a sink that can never trip: |numerator|^2 = r0^2 - y r1^2 is a sum of non-negative terms, and
                                            the sign of the TRUNCATED E(y) is masked off -- the plan validates it only where a spec
                                            looks, and beyond the last band it may well go negative (found by tools/fuzz_parity.py: it
                                            used to fail spec 0 on such samples) */
    int gi = 0;
    for (int rn = 0; rn < Q.nplain; rn++) {
        const unsigned int any = Q.runs[rn].any, all = Q.runs[rn].all;
        if (Q.runs[rn].g0 != gi) {       /* a fused run was taken out in front of this one: the preloaded grid values are not its */
            gi = Q.runs[rn].g0;
#pragma unroll
            for (int h = 0; h < PT; h += 2) { const double2 a = __ldg((const double2 *)(Q.y1 + gi * PT + h)); y[h] = a.x; y[h + 1] = a.y; }
        }
        const int g_end = gi + Q.runs[rn].ngroups;
        const int one = (any == all && all != 0u && (all & (all - 1u)) == 0u) ? __ffs((int)all) - 1 : -1;
        if (any == 0u) {
            for (; gi < g_end; gi++) { QO_TS_CORE QO_PTS_N(PT) idle |= tf_hi(n2[p]) | (tf_hi(dd[p]) & 0x7fffffffu); }
        } else if (one >= 0 && one == hs) {
            for (; gi < g_end; gi++) {
                QO_TS_CORE
                QO_TS_VALUE
                trkv = hneg ? tf_extreme<PT, true>(val, trkv) : tf_extreme<PT, false>(val, trkv);
            }
        } else if (one >= 0) {
            unsigned int a1 = 0u;
            if (P.neg[one]) { const double t = -P.thr[one]; for (; gi < g_end; gi++) { QO_TS_CORE QO_PTS_N(PT) a1 |= tf_hi(fma(t, dd[p], n2[p])); } }
            else { const double t = P.thr[one]; for (; gi < g_end; gi++) { QO_TS_CORE QO_PTS_N(PT) a1 |= tf_hi(fma(t, dd[p], -n2[p])); } }
#pragma unroll
            for (int sp = 0; sp < NS; sp++) if (sp == one) acc[sp] |= a1;
        } else {
            /* several specs at once, or a group that straddles a band edge (per-point byte masks) */
            for (; gi < g_end; gi++) {
                QO_TS_CORE
                unsigned int mwv[PT];
                if (any != all) { QO_PTS_N(PT) mwv[p] = __ldg(&Q.mw[j + p].x); }
                else { QO_PTS_N(PT) mwv[p] = 0xffffffffu; }
#pragma unroll
                for (int sp = 0; sp < NS; sp++) {
                    if (!((any >> sp) & 1u)) continue;
                    if (sp == hs) {
                        QO_TS_VALUE
                        QO_PTS_N(PT) { const bool in = (mwv[p] >> (8 * sp)) & 1u; val[p] = in ? val[p] : (hneg ? 1.7e308 : -1.7e308); }
                        trkv = hneg ? tf_extreme<PT, true>(val, trkv) : tf_extreme<PT, false>(val, trkv);
                    } else if (P.neg[sp]) { const double t = -P.thr[sp]; QO_PTS_N(PT) acc[sp] |= tf_hi(fma(t, dd[p], n2[p])) & __byte_perm(mwv[p], 0, 0x1111 * sp); }
                    else { const double t = P.thr[sp]; QO_PTS_N(PT) acc[sp] |= tf_hi(fma(t, dd[p], -n2[p])) & __byte_perm(mwv[p], 0, 0x1111 * sp); }
                }
            }
        }
    }
#undef QO_TS_VALUE
#undef QO_TS_CORE
    /* the fused runs (plain ladders only): one spec active, its margin sg (N2 - t E) one polynomial of NF coefficients formed
     * once per sample (qo_tf_fuse) -- one Horner chain per point instead of three chains, |.|^2 and the margin.  cn and ce are
     * dead from here on: the polynomial takes their registers */
    if constexpr (NN == 2) {
        if (Q.nplain < Q.nruns) {                        /* none for most jobs */
            constexpr int NF = 2 * KN > KE ? 2 * KN : KE;
            const int one = __ffs((int)Q.runs[Q.nplain].all) - 1;
            double fz[NF];
            qo_tf_fuse(KN, KE, cn, ce, P.thr[one], P.neg[one], fz);
            unsigned int a1 = 0u;
            constexpr int PF = QO_TS_FG2 * PT;
            double yf[PF];
            for (int rn = Q.nplain; rn < Q.nruns; rn++) {
                gi = Q.runs[rn].g0;
                const int g_end = gi + Q.runs[rn].ngroups;
#pragma unroll
                for (int h = 0; h < PF; h += 2) { const double2 a = __ldg((const double2 *)(Q.y1 + gi * PT + h)); yf[h] = a.x; yf[h + 1] = a.y; }
                for (; gi + QO_TS_FG2 <= g_end; gi += QO_TS_FG2) {
                    double F[PF];
                    QO_PTS_N(PF) F[p] = fma(fz[NF - 1], yf[p], fz[NF - 2]);
#pragma unroll
                    for (int m = NF - 3; m >= 0; m--) { QO_PTS_N(PF) F[p] = fma(F[p], yf[p], fz[m]); }
#pragma unroll
                    for (int h = 0; h < PF; h += 2) { const double2 a = __ldg((const double2 *)(Q.y1 + (gi + QO_TS_FG2) * PT + h)); yf[h] = a.x; yf[h + 1] = a.y; }
                    QO_PTS_N(PF) a1 |= tf_hi(F[p]);
                }
                for (; gi < g_end; gi++) {                /* the run's last groups: yf[0, PT) holds the next one */
                    double F[PT];
                    QO_PTS_N(PT) F[p] = fma(fz[NF - 1], yf[p], fz[NF - 2]);
#pragma unroll
                    for (int m = NF - 3; m >= 0; m--) { QO_PTS_N(PT) F[p] = fma(F[p], yf[p], fz[m]); }
#pragma unroll
                    for (int h = 0; h < PT; h += 2) { const double2 a = __ldg((const double2 *)(Q.y1 + (gi + 1) * PT + h)); yf[h] = a.x; yf[h + 1] = a.y; }
                    QO_PTS_N(PT) a1 |= tf_hi(F[p]);
                }
            }
#pragma unroll
            for (int sp = 0; sp < NS; sp++) if (sp == one) acc[sp] |= a1;
        }
    }
    if (idle >> 31) acc[0] |= idle;      /* never taken (see above); keeps the unobserved points' arithmetic alive */
}

/* the body for this launch's (kn, kd): one switch per launch, outside the frequency loop */
#ifdef QO_TS_DEV_KN          /* development builds: a few loop bodies only */
#define QO_TS_KN_OK(k) ((k) == QO_TS_DEV_KN || (k) == QO_TS_DEV_KN2)
#define QO_TS_KE_OK(k) ((k) == QO_TS_DEV_KE || (k) == QO_TS_DEV_KE2)
#else
#define QO_TS_KN_OK(k) true
#define QO_TS_KE_OK(k) true
#endif
/* the loop body for this launch's kd (KN is the kernel's): one switch per sample, outside the frequency loop */
template <int NN, int KN, bool CPL, int NS, int PT>
__device__ __forceinline__ void ts_pick_e(const TsParams &Q, unsigned long long sample, unsigned int (&acc)[NS], double &trkv)
{
    constexpr int CAPE = NN == 2 ? QO_TS_CAPE2 : QO_TS_CAPE4;
    const int kd = Q.t.den == QO_TF_DEN_E ? Q.t.kd : 0;
#define QO_TS_CASE(K) case K: if (K <= CAPE && QO_TS_KE_OK(K)) ts_loop<NN, KN, (K <= CAPE ? K : 0), CPL, NS, PT>(Q, sample, acc, trkv); break;
#ifdef QO_TS_DEV_KN
    if (!QO_TS_KN_OK(KN) || !QO_TS_KE_OK(kd)) __trap();          /* a development build was asked for a body it does not carry */
#endif
    switch (kd) {
        QO_TS_CASE(0) QO_TS_CASE(2) QO_TS_CASE(4) QO_TS_CASE(6) QO_TS_CASE(8) QO_TS_CASE(10) QO_TS_CASE(12) QO_TS_CASE(14) QO_TS_CASE(16)
    default: __trap();                                            /* qo_ts_eligible admits only the lengths above */
    }
#undef QO_TS_CASE
}

template <int NN, bool CPL, int PT, int MINB, int KN>
__global__ void __launch_bounds__(QO_TS_TPB, MINB) qo_mc_ts_kernel(const __grid_constant__ TsParams Q)
{
    constexpr int NS = 4;
    static_assert(NN == 2 || NN == 4, "two or four numerator chains");
    static_assert(CPL == (NN == 4), "P and Q stay apart exactly when a coupled-line block is in front");
    const TfParams &P = Q.t;
    __shared__ unsigned int s_cnt[2 + QO_NSPEC_MAX + QO_MAX_HIST];
    const int lane = threadIdx.x & 31;
    const int ncnt = 2 + P.nspec + (P.hist_bins > 0 ? P.hist_bins : 0);
    for (int i = threadIdx.x; i < ncnt; i += QO_TS_TPB) s_cnt[i] = 0;
    __syncthreads();
    const int hs = P.hist_spec;
    const bool hneg = hs >= 0 && P.neg[hs & (QO_TF_NSPEC - 1)];
    /* a warp takes 32 consecutive samples at a time, the first batch by position, the following ones from a ticket counter: the
     * work per sample is identical, but the issue scheduler is not fair -- with a static deal the favoured warps finish early
     * and an SM sub-partition averages 2.9 of its 4 warps (ncu), with tickets all four stay busy to the end */
    const unsigned long long nwarps = (unsigned long long)gridDim.x * (QO_TS_TPB / 32);
    unsigned long long batch = (unsigned long long)blockIdx.x * (QO_TS_TPB / 32) + (threadIdx.x >> 5);
    while (batch < Q.nbatches) {
        unsigned long long next = 0;
        if (lane == 0) next = nwarps + atomicAdd(Q.ticket, 1ull);
        const unsigned long long sample = batch * 32ull + (unsigned long long)lane;
        unsigned int acc[NS];
#pragma unroll
        for (int sp = 0; sp < NS; sp++) acc[sp] = 0u;
        double trkv = hneg ? 1.7e308 : -1.7e308;
        ts_pick_e<NN, KN, CPL, NS, PT>(Q, sample, acc, trkv);
        /* stage D: verdict per thread */
        unsigned int fail = 0;
#pragma unroll
        for (int sp = 0; sp < NS; sp++)
            if (sp < P.nspec && sp != hs && (acc[sp] >> 31)) fail |= 1u << sp;
        if (hs >= 0) {
            const double t = P.thr[hs & (QO_TF_NSPEC - 1)];
            if (hneg ? trkv < t : trkv > t) fail |= 1u << hs;
        }
        const unsigned int okm = __ballot_sync(0xffffffffu, fail == 0u);
        if (lane == 0) { atomicAdd(&s_cnt[0], (unsigned int)__popc(okm)); atomicAdd(&s_cnt[1], 32u); }
        for (int sp = 0; sp < P.nspec; sp++) {
            const unsigned int m = __ballot_sync(0xffffffffu, (fail >> sp) & 1u);
            if (lane == 0 && m) atomicAdd(&s_cnt[2 + sp], (unsigned int)__popc(m));
        }
        if (hs >= 0) {
            const double k21 = P.k21;
            const double lin = hneg ? k21 * k21 * (1.0 / trkv) : k21 * k21 / trkv;
            const double v = 10.0 * log10(lin);
            const double xb = (v - P.hist_lo) / (P.hist_hi - P.hist_lo) * (double)P.hist_bins;
            long long bin = (long long)floor(xb);
            if (!(xb >= 0.0)) bin = 0;
            if (bin >= P.hist_bins) bin = P.hist_bins - 1;
            atomicAdd(&s_cnt[2 + P.nspec + (int)bin], 1u);
        }
        batch = __shfl_sync(0xffffffffu, next, 0);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < ncnt; i += QO_TS_TPB)
        if (s_cnt[i]) atomicAdd(&P.counters[i], (unsigned long long)s_cnt[i]);
}
