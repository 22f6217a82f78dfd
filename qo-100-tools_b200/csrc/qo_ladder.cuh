/*
 * qo_ladder.cuh -- the straight-line Monte-Carlo kernel for the pcb/generic-filter
 * ladder family (reference: pcb/generic-filter/README.md:13 "up to 11th order",
 * qo-100-generic-filter.sch:1450-1488,1703-1995 -- alternating series / shunt
 * branches), optionally preceded by the coupled-line through section of
 * util/directional-couplers/<name>.trc (BASELINE configs 2 and 5).  sm_100a only.
 *
 * Why a second kernel next to the opcode interpreter of qo_lumped.cuh: ncu on the
 * interpreter (profiles/r01a_*) shows the FP64 pipe 47 % busy with 53 % of the
 * issued instructions being dispatch overhead (BRA/ISETP/IMAD.MOV/LDS) and the
 * dominant stall a fixed-latency wait on the serial immittance -> reciprocal ->
 * chain dependency of ONE element.  Here the element sequence is a template
 * parameter, so the whole ladder is one basic block: ptxas overlaps the
 * reciprocal of element k+1 with the chain update of element k, and the only
 * non-FP64 work left is the broadcast LDS of the per-sample coefficients.
 *
 * Arithmetic (all FP64, one thread = PTS (sample, frequency) points of ONE sample):
 *   |S21|^2 = 4 Rs Rl / |den|^2,  den = [1 Rs] . M1 M2 ... MN . [Rl 1]^T
 * Reduce-only specs on |S21| need den only, so the chain carries the ROW VECTOR
 * u = [1 Rs] . M1 ... Mk = (a, b) instead of the 2x2 product (half the FMAs):
 *   series Z: b += a Z        shunt Y: a += b Y        den = a Rl + b
 * Jobs with |S11| specs add the second row vector v = [1 -Rs] . M1 ... Mk (NROWS = 2):
 *   S11 = (v . [Rl 1]^T) / den
 * Series lossy inductor (R + jwL) || 1/(jwCp), with D = 1 - w^2 L Cp:
 *   Z = (R + j w (L D - R^2 Cp)) / (D^2 + w^2 (R Cp)^2)       [numerator real part is exactly R]
 * Shunt lossy capacitor R + jwLs + 1/(jwC), X = w Ls - (1/w)(1/C):
 *   Y = (R - jX) / (R^2 + X^2)
 * Executed FP64 instructions per eval for the 11th-order ladder: 6*15 + 5*12 - 3
 * (first step) + 4 (den, |den|^2) + nspec compares = 151 + nspec (DESIGN.md).
 *
 * Spec bookkeeping: per spec one running extreme of |den|^2 over the spec's band
 * (sign-flipped for "max dB" specs so that every tracker is a running MAX),
 * compared with the threshold once per sample; the histogram variable is the
 * tracker of its spec, so it costs nothing extra.
 */
#pragma once
#include "qo_lumped.cuh"

#define QO_LAD_MAXN 11
#define QO_LAD_NSPEC 4               /* trackers kept in registers; more specs -> interpreter */
#define QO_LAD_STRIDE 6              /* values per element record (16-byte aligned in FP64, 8-byte in FP32) */
#define QO_LAD_CPL 10                /* values of the coupler record that precedes the ladder records */

/* The kernel is generic over T = double (the product's precision, every number quoted in DESIGN.md) and
 * T = float (the optional FP32 mode of north_star: |S21| within 1e-3 dB, on the 2x wider FP32 pipe). */
template <typename T> struct LadNum;
template <> struct LadNum<double> { static __device__ __forceinline__ double neg_huge() { return -1.7e308; } };
template <> struct LadNum<float> { static __device__ __forceinline__ float neg_huge() { return -3.0e38f; } };

/* NROWS = 1: the row vector u = [1 Rs] M (enough for |S21|); NROWS = 2 adds v = [1 -Rs] M, whose contraction
 * v . [Rl 1]^T is the numerator of S11, for jobs with |S11| specs */
template <typename T, int PTS, int NROWS> struct LadRow { T ar[NROWS][PTS], ai[NROWS][PTS], br[NROWS][PTS], bi[NROWS][PTS]; };
#define QO_ROWS _Pragma("unroll") for (int r = 0; r < NROWS; r++)
#define QO_PTS _Pragma("unroll") for (int p = 0; p < PTS; p++)

/* Broadcast read of two coefficients from the warp's record table.  The records are invariant over
 * the frequency loop, and left to itself ptxas hoists all 55 values of an 11-element ladder out of
 * the loop and spills them to local memory; an asm volatile load stays where it is written (one
 * conflict-free wavefront per load). */
template <typename T> struct LadV2 { T x, y; };
__device__ __forceinline__ LadV2<double> lad_lds2(unsigned int saddr, double)
{
    LadV2<double> v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(saddr));
    return v;
}
__device__ __forceinline__ LadV2<float> lad_lds2(unsigned int saddr, float)
{
    LadV2<float> v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(saddr));
    return v;
}
__device__ __forceinline__ double lad_lds1(unsigned int saddr, double)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ float lad_lds1(unsigned int saddr, float)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(saddr));
    return v;
}

/* 1/q for the PTS points of one element.
 * FP64: ONE reciprocal for all points (Montgomery's trick): the MUFU.RCP64H seed and the register move that
 * zeroes its low word are not FP64-pipe instructions, and tools/pipe_probe2.cu shows each such instruction costs
 * about one FP64 issue cycle when it does not land in a DFMA's shadow.  FP64 work is unchanged (9 DMUL + 3 DFMA
 * per four points = 3 per point); each 1/q carries <= 3 roundings.  The product of four |immittance|^2 values
 * stays far inside the double range for any physical element.
 * FP32: one MUFU.RCP per point (1 ulp; a product of four would leave the float range). */
template <int PTS> __device__ __forceinline__ void lad_rcp_batch(const double (&q)[PTS], double (&s)[PTS])
{
    static_assert(PTS == 2 || PTS % 4 == 0, "two points or a multiple of four points per thread");
    if (PTS > 4) {                       /* batches of four */
#pragma unroll
        for (int h = 0; h < PTS; h += 4) {
            const double p01 = q[h] * q[h + 1], p23 = q[h + 2] * q[h + 3];
            const double r = qrcp(p01 * p23);
            const double r01 = r * p23, r23 = r * p01;
            s[h] = r01 * q[h + 1]; s[h + 1] = r01 * q[h]; s[h + 2] = r23 * q[h + 3]; s[h + 3] = r23 * q[h + 2];
        }
    } else if (PTS == 2) {
        const double r = qrcp(q[0] * q[1]);
        s[0] = r * q[1]; s[1] = r * q[0];
    } else {
        const double p01 = q[0] * q[1], p23 = q[2] * q[3];
        const double r = qrcp(p01 * p23);
        const double r01 = r * p23, r23 = r * p01;
        s[0] = r01 * q[1]; s[1] = r01 * q[0]; s[2] = r23 * q[3]; s[3] = r23 * q[2];
    }
}
template <int PTS> __device__ __forceinline__ void lad_rcp_batch(const float (&q)[PTS], float (&s)[PTS])
{
    QO_PTS asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(s[p]) : "f"(q[p]));
}

/* series lossy inductor; record = { L*Cp, (R*Cp)^2, L, R^2*Cp, R, - } */
template <typename T, int PTS, int NROWS, bool FIRSTSTEP>
__device__ __forceinline__ void lad_ser_lossy_l(unsigned int cf, const T (&w)[PTS], const T (&w2)[PTS], T rs, LadRow<T, PTS, NROWS> &u)
{
    const LadV2<T> c01 = lad_lds2(cf, T()), c23 = lad_lds2(cf + 2 * sizeof(T), T());
    const T R = lad_lds1(cf + 4 * sizeof(T), T());
    T dre[PTS], q[PTS], s[PTS];
    QO_PTS { dre[p] = qfma(-w2[p], c01.x, T(1)); q[p] = qfma(dre[p], dre[p], w2[p] * c01.y); }
    lad_rcp_batch<PTS>(q, s);
    QO_PTS {
        const T g = qfma(c23.x, dre[p], -c23.y);
        const T zr = R * s[p], zi = (w[p] * s[p]) * g;
        QO_ROWS {
            if (FIRSTSTEP) {             /* u = [1 +-Rs]: b = +-Rs + Z */
                u.br[r][p] = (r ? -rs : rs) + zr; u.bi[r][p] = zi;
            } else {
                u.br[r][p] = qfma(u.ar[r][p], zr, u.br[r][p]); u.br[r][p] = qfma(-u.ai[r][p], zi, u.br[r][p]);
                u.bi[r][p] = qfma(u.ar[r][p], zi, u.bi[r][p]); u.bi[r][p] = qfma(u.ai[r][p], zr, u.bi[r][p]);
            }
        }
    }
}

/* shunt lossy capacitor; record = { 1/C, Ls, R, R^2 } */
template <typename T, int PTS, int NROWS, bool FIRSTSTEP>
__device__ __forceinline__ void lad_shunt_lossy_c(unsigned int cf, const T (&w)[PTS], const T (&wi)[PTS], T rs, LadRow<T, PTS, NROWS> &u)
{
    const LadV2<T> c01 = lad_lds2(cf, T()), c23 = lad_lds2(cf + 2 * sizeof(T), T());
    T x[PTS], q[PTS], s[PTS];
    QO_PTS { x[p] = qfma(w[p], c01.y, -wi[p] * c01.x); q[p] = qfma(x[p], x[p], c23.y); }
    lad_rcp_batch<PTS>(q, s);
    QO_PTS {
        const T yr = c23.x * s[p], yi = -x[p] * s[p];
        QO_ROWS {
            if (FIRSTSTEP) {             /* u = [1 +-Rs]: a = 1 +- Rs Y */
                const T rr = r ? -rs : rs;
                u.ar[r][p] = qfma(rr, yr, T(1)); u.ai[r][p] = rr * yi;
            } else {
                u.ar[r][p] = qfma(u.br[r][p], yr, u.ar[r][p]); u.ar[r][p] = qfma(-u.bi[r][p], yi, u.ar[r][p]);
                u.ai[r][p] = qfma(u.br[r][p], yi, u.ai[r][p]); u.ai[r][p] = qfma(u.bi[r][p], yr, u.ai[r][p]);
            }
        }
    }
}

/* Coupled-line through section as the FIRST block (SURVEY App. B.4), division-free.
 * Mode lines normalised to Zt: D_m = 2 cos(t_m) + j sin(t_m) (z_m + 1/z_m), n_m = j sin(t_m) (z_m - 1/z_m);
 * S21 = Sg/Pi, S11 = Nu/Pi with Pi = D_e D_o, Sg = D_e + D_o, Nu = (n_e D_o + n_o D_e)/2.  Symmetric S -> ABCD:
 *   A = (Pi^2 - Nu^2 + Sg^2)/k,  B = Zt ((Pi + Nu)^2 - Sg^2)/k,  C = ((Pi - Nu)^2 - Sg^2)/(Zt k),  k = 2 Sg Pi.
 * The complex scalar 1/k multiplies the whole matrix, hence den, so the chain runs on k*[A B; C A] and
 * |den|^2 is rescaled by 1/|k|^2 at the end (one batched real reciprocal instead of three complex divides).
 * record = { z_e + 1/z_e, (z_e - 1/z_e)/2, (odd: same two), te/w, to/w, Zt, Rs/Zt, te/w - nominal, to/w - nominal }
 *
 * Angles: t_m = k_m w.  When the plan could bound the perturbation |k_m - k_m,nominal| w_max <= 0.1 rad
 * (FAST), sin/cos of the NOMINAL angle come from per-frequency tables and the sample's small rotation from
 * short Taylor polynomials (truncation |d|^10/10! < 3e-17 on cos, |d|^9/9! < 3e-15 on sin) -- 14 FP64 instructions instead of the ~30 of
 * a general sincos; otherwise sincos() is called. */
/* mode angles of the coupler block for the PTS points: sin/cos of t_e = k_e w and t_o = k_o w (record layout as above) */
template <typename T, int PTS, bool FAST>
__device__ __forceinline__ void lad_cpl_angles(unsigned int cf, const T (&w)[PTS], const T (&tse)[PTS], const T (&tce)[PTS],
                                               const T (&tso)[PTS], const T (&tco)[PTS], T (&se)[PTS], T (&ce)[PTS], T (&so)[PTS], T (&co)[PTS])
{
    const LadV2<T> c45 = lad_lds2(cf + 4 * sizeof(T), T()), c89 = lad_lds2(cf + 8 * sizeof(T), T());
    const T ke = c45.x, ko = c45.y;
    const bool same = ke == ko;
    QO_PTS {
        if (FAST) {
            {
                const T d = c89.x * w[p], z = d * d;
                const T cd = qfma(qfma(qfma(qfma(T(1.0 / 40320.0), z, T(-1.0 / 720.0)), z, T(1.0 / 24.0)), z, T(-0.5)), z, T(1));
                const T sd = d * qfma(qfma(qfma(T(-1.0 / 5040.0), z, T(1.0 / 120.0)), z, T(-1.0 / 6.0)), z, T(1));
                se[p] = qfma(tse[p], cd, tce[p] * sd); ce[p] = qfma(tce[p], cd, -tse[p] * sd);
            }
            if (same) { so[p] = se[p]; co[p] = ce[p]; }
            else {
                const T d = c89.y * w[p], z = d * d;
                const T cd = qfma(qfma(qfma(qfma(T(1.0 / 40320.0), z, T(-1.0 / 720.0)), z, T(1.0 / 24.0)), z, T(-0.5)), z, T(1));
                const T sd = d * qfma(qfma(qfma(T(-1.0 / 5040.0), z, T(1.0 / 120.0)), z, T(-1.0 / 6.0)), z, T(1));
                so[p] = qfma(tso[p], cd, tco[p] * sd); co[p] = qfma(tco[p], cd, -tso[p] * sd);
            }
        } else {
            qsincos(ke * w[p], &se[p], &ce[p]);
            if (same) { so[p] = se[p]; co[p] = ce[p]; } else qsincos(ko * w[p], &so[p], &co[p]);
        }
    }
}

template <typename T, int PTS, int NROWS, bool FAST, bool RAWK = false>
__device__ __forceinline__ void lad_cpl_first(unsigned int cf, const T (&w)[PTS], const T (&tse)[PTS], const T (&tce)[PTS],
                                              const T (&tso)[PTS], const T (&tco)[PTS], T rs, LadRow<T, PTS, NROWS> &u, T (&scale)[PTS])
{
    const LadV2<T> c01 = lad_lds2(cf, T()), c23 = lad_lds2(cf + 2 * sizeof(T), T()), c67 = lad_lds2(cf + 6 * sizeof(T), T());
    const T cE = c01.x, hE = c01.y, cO = c23.x, hO = c23.y, zt = c67.x, rz = c67.y;
    T se[PTS], ce[PTS], so[PTS], co[PTS], kap2[PTS];
    lad_cpl_angles<T, PTS, FAST>(cf, w, tse, tce, tso, tco, se, ce, so, co);
    QO_PTS {
        const T a1 = ce[p] + ce[p], b1 = se[p] * cE, a2 = co[p] + co[p], b2 = so[p] * cO;             /* D_e, D_o */
        const T Pr = qfma(a1, a2, -b1 * b2), Pi = qfma(a1, b2, a2 * b1);                                 /* Pi */
        const T Sr = a1 + a2, Si = b1 + b2;                                                              /* Sg */
        const T pe = se[p] * hE, po = so[p] * hO;
        const T Nr = -qfma(pe, b2, po * b1), Ni = qfma(pe, a2, po * a1);                                 /* Nu */
        const T Xr = qfma(Pr, Pr, -Pi * Pi), Xi = (Pr + Pr) * Pi;                                        /* Pi^2 */
        const T Yr = qfma(Nr, Nr, -Ni * Ni), Yi = (Nr + Nr) * Ni;                                        /* Nu^2 */
        const T Wr = qfma(Sr, Sr, -Si * Si), Wi = (Sr + Sr) * Si;                                        /* Sg^2 */
        const T Vr = qfma(Pr, Nr, -Pi * Ni), Vi = qfma(Pr, Ni, Pi * Nr);                                 /* Pi Nu */
        const T Tr = Xr + Yr - Wr, Ti = Xi + Yi - Wi;
        const T Ar = Xr - Yr + Wr, Ai = Xi - Yi + Wi;                                                    /* k A */
        const T Br = qfma(T(2), Vr, Tr), Bi = qfma(T(2), Vi, Ti);                                        /* k B / Zt */
        const T Cr = qfma(T(-2), Vr, Tr), Ci = qfma(T(-2), Vi, Ti);                                      /* k C Zt */
        const T Kr = qfma(Sr, Pr, -Si * Pi), Ki = qfma(Sr, Pi, Si * Pr);                                 /* k / 2 */
        kap2[p] = qfma(Kr, Kr, Ki * Ki);
        QO_ROWS {
            const T sg = r ? T(-1) : T(1);
            u.ar[r][p] = qfma(sg * rz, Cr, Ar); u.ai[r][p] = qfma(sg * rz, Ci, Ai);                      /* k (A +- Rs C) */
            u.br[r][p] = qfma(sg * rs, Ar, zt * Br); u.bi[r][p] = qfma(sg * rs, Ai, zt * Bi);            /* k (B +- Rs A) */
        }
    }
    if (RAWK) { QO_PTS scale[p] = T(4) * kap2[p]; }                                                      /* |k|^2: the caller folds it into its own denominator */
    else {
        lad_rcp_batch<PTS>(kap2, scale);
        QO_PTS scale[p] *= T(0.25);                                                                      /* 1/|k|^2 */
    }
}

/* per-sample coefficient records, one lane per element (perturbation is the shared bit-exact stream; the
 * derived coefficients are formed in FP64 and rounded once when T = float) */
template <typename T>
__device__ __forceinline__ void lad_derive(const DevProg *__restrict__ prog, int e, const double *__restrict__ x, T *out,
                                           const double *__restrict__ cplms, double *nom_k)
{
    double p[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        p[k] = prog->nom[e][k];
        const int tv = prog->tvar[e][k];
        if (tv >= 0) p[k] = qo_stream_apply(p[k], prog->ttol[e][k], x[tv], prog->tmode[e][k]);
    }
    nom_k[0] = prog->nom[e][2] / (360.0 * prog->nom[e][4]); nom_k[1] = prog->nom[e][3] / (360.0 * prog->nom[e][4]);
    if (e == prog->cplms_elem) {
        /* physical coupled line: p[] holds (W, S, L, H_t, f0, Zt); this sample's electrical view comes from the pre-pass */
        p[0] = cplms[0]; p[1] = cplms[1]; p[2] = cplms[2]; p[3] = cplms[3]; p[4] = prog->nom[e][4]; p[5] = prog->nom[e][5];
        nom_k[0] = prog->cplms_nom[2] / (360.0 * p[4]); nom_k[1] = prog->cplms_nom[3] / (360.0 * p[4]);
    }
    switch (prog->opcode[e]) {
    case OP_SER_LOSSY_L: case OP_SER_L: {              /* p = L, R, Cp */
        const double rcp_ = p[1] * p[2];
        out[0] = T(p[0] * p[2]); out[1] = T(rcp_ * rcp_); out[2] = T(p[0]); out[3] = T(p[1] * rcp_); out[4] = T(p[1]); out[5] = T(0);
        break;
    }
    case OP_SHUNT_LOSSY_C: case OP_SHUNT_C:            /* p = C, R, Ls */
        out[0] = T(1.0 / p[0]); out[1] = T(p[2]); out[2] = T(p[1]); out[3] = T(p[1] * p[1]); out[4] = T(0); out[5] = T(0);
        break;
    case OP_CPL: {
        const double a = p[0] / p[5], b = p[1] / p[5];
        const double ke = p[2] / (360.0 * p[4]), ko = p[3] / (360.0 * p[4]);
        out[0] = T(a + 1.0 / a); out[1] = T(0.5 * (a - 1.0 / a)); out[2] = T(b + 1.0 / b); out[3] = T(0.5 * (b - 1.0 / b));
        out[4] = T(ke); out[5] = T(ko); out[6] = T(p[5]); out[7] = T(prog->rs / p[5]);
        out[8] = T(ke - nom_k[0]); out[9] = T(ko - nom_k[1]);
        break;
    }
    default: break;
    }
}

/* everything warp-uniform travels as a kernel parameter (constant bank -> uniform registers, no
 * vector registers held across the frequency loop) */
struct LadParams {
    const DevProg *prog;
    const void *wt, *wit, *wsqt;             /* w, 1/w, w^2 per grid point, two points per entry (double2 / float2) */
    const uchar2 *m2;                        /* per-point spec bit masks */
    const void *cse, *cce, *cso, *cco;       /* coupler: sin/cos of the NOMINAL even/odd angle per grid point (cpl_fast) */
    unsigned long long *counters;
    unsigned long long *ticket;              /* next unclaimed sample of this launch (zeroed on the stream before it) */
    unsigned long long sample_offset, nsamples, seed;
    double rs, rl, k21, hist_lo, hist_hi;
    double thr[QO_LAD_NSPEC];                /* sign-adjusted thresholds: FAIL iff tracker > thr */
    int neg[QO_LAD_NSPEC];                   /* "max dB" spec: the tracker holds -|den|^2 */
    int is_s11[QO_LAD_NSPEC];                /* the spec's tracker holds |S11|^2 = |n11|^2 / |den|^2 (NROWS == 2 kernels) */
    int npairs, n_var, n_ops, nspec, dist, hist_spec, hist_bins, hist_kind;
    int cpl_fast, cpl_same;                  /* small-angle table path usable; nominal even and odd angles identical */
    int op0;                                 /* first op of the chain (leading OP_NOPs: a substrate that only serves a QO_CPL_MS) */
    const double *cplms;                     /* physical coupled line: per-sample Z0e, Z0o, theta_e, theta_o (pre-pass) */
};

/*
 * T      double | float                 N      ladder elements (1..11)
 * FIRST  0 = series element first, 1 = shunt first            CPL    coupled-line block in front
 * NROWS  1 | 2 (with the |S11| row)     PP     frequency pairs per thread per iteration (PTS = 2*PP points)
 * TPB / MINB  block size and resident blocks per SM (register budget = 65536 / (TPB*MINB))
 * One warp = one sample at a time; lane l owns pairs l, l+32, ... of that sample's grid.
 * Samples are handed out through a global ticket counter: with a static split ncu showed every
 * SMSP averaging 3.06 of its 4 warps (the issue scheduler is not fair, favoured warps finished
 * their share early and the FP64 pipe drained); tickets keep all warps busy until the pool is empty.
 */
template <typename T, int N, int FIRST, bool CPL, int NROWS, int PP, int TPB, int MINB>
__global__ void __launch_bounds__(TPB, MINB) qo_mc_ladder_kernel(const __grid_constant__ LadParams P)
{
    typedef typename QoVec2<T>::type V2;
    constexpr int PTS = 2 * PP;
    constexpr int WARPS = TPB / 32;
    constexpr int NREC = (CPL ? QO_LAD_CPL : 0) + N * QO_LAD_STRIDE;
    __shared__ __align__(16) T s_coef[WARPS][NREC];
    __shared__ double s_x[WARPS][QO_MAX_VAR];
    __shared__ unsigned int s_cnt[QO_NCNT_MAX];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ncnt = qo_ncnt(P.nspec, P.hist_bins);
    qo_tally_zero<TPB>(s_cnt, ncnt);
    __syncthreads();

    T *coefw = s_coef[warp];
    double *xw = s_x[warp];
    const unsigned int coefs = (unsigned int)__cvta_generic_to_shared(coefw);
    const int npairs = P.npairs;
    const T rs = T(P.rs);
    const V2 *wt = (const V2 *)P.wt, *wit = (const V2 *)P.wit, *wsqt = (const V2 *)P.wsqt;

    /* the first gridDim.x*WARPS samples are claimed by position, the rest by ticket; the next ticket
     * is requested before the frequency loop so that the atomic's latency is never exposed */
    const unsigned long long total_warps = (unsigned long long)gridDim.x * WARPS;
    unsigned long long s = (unsigned long long)blockIdx.x * WARPS + warp;
    while (s < P.nsamples) {
        unsigned long long s_next = 0;
        if (lane == 0) s_next = total_warps + atomicAdd(P.ticket, 1ull);
        /* 1. the sample's random variables (Philox, counter-based) and coefficient records */
        for (int v = lane; v < P.n_var; v += 32) xw[v] = qo_stream_variate(P.seed, P.sample_offset + s, (uint32_t)v, P.dist);
        __syncwarp();
        if (lane + P.op0 < P.n_ops) {
            const int rec = CPL ? (lane == 0 ? 0 : QO_LAD_CPL + (lane - 1) * QO_LAD_STRIDE) : lane * QO_LAD_STRIDE;
            double nom_k[2];
            lad_derive<T>(P.prog, lane + P.op0, xw, coefw + rec, P.cplms ? P.cplms + 4 * s : NULL, nom_k);
        }
        __syncwarp();

        /* 2. frequency loop */
        T trk[QO_LAD_NSPEC];
#pragma unroll
        for (int sp = 0; sp < QO_LAD_NSPEC; sp++) trk[sp] = LadNum<T>::neg_huge();       /* "no point seen yet" */
        /* warp-uniform trip count (the tracker vote below is a full-warp collective): lanes past the end of
         * the grid re-evaluate the last pair with all-zero masks */
        for (int jb = 0; jb < npairs; jb += 32 * PP) {
            const int j0 = jb + lane;
            T w[PTS], wi[PTS], w2[PTS];
            unsigned int mk[PTS];
#pragma unroll
            for (int q = 0; q < PP; q++) {
                const int j = j0 + 32 * q;
                const int jc = j < npairs ? j : npairs - 1;
                const V2 a = wt[jc], b = wit[jc], c = wsqt[jc];
                const uchar2 m = P.m2[jc];
                w[2 * q] = a.x; w[2 * q + 1] = a.y; wi[2 * q] = b.x; wi[2 * q + 1] = b.y; w2[2 * q] = c.x; w2[2 * q + 1] = c.y;
                mk[2 * q] = j < npairs ? m.x : 0u; mk[2 * q + 1] = j < npairs ? m.y : 0u;
            }
            LadRow<T, PTS, NROWS> u;
            T cscale[PTS];
            QO_PTS { cscale[p] = T(1); QO_ROWS { u.ar[r][p] = T(1); u.ai[r][p] = T(0); u.br[r][p] = r ? -rs : rs; u.bi[r][p] = T(0); } }
            if (CPL) {
                T tse[PTS], tce[PTS], tso[PTS], tco[PTS];
                QO_PTS { tse[p] = T(0); tce[p] = T(1); tso[p] = T(0); tco[p] = T(1); }
                if (P.cpl_fast) {
#pragma unroll
                    for (int q = 0; q < PP; q++) {
                        const int j = j0 + 32 * q;
                        const int jc = j < npairs ? j : npairs - 1;
                        const V2 a = ((const V2 *)P.cse)[jc], b = ((const V2 *)P.cce)[jc];
                        tse[2 * q] = a.x; tse[2 * q + 1] = a.y; tce[2 * q] = b.x; tce[2 * q + 1] = b.y;
                        if (!P.cpl_same) {
                            const V2 c = ((const V2 *)P.cso)[jc], d = ((const V2 *)P.cco)[jc];
                            tso[2 * q] = c.x; tso[2 * q + 1] = c.y; tco[2 * q] = d.x; tco[2 * q + 1] = d.y;
                        }
                    }
                    lad_cpl_first<T, PTS, NROWS, true>(coefs, w, tse, tce, tso, tco, rs, u, cscale);
                } else {
                    lad_cpl_first<T, PTS, NROWS, false>(coefs, w, tse, tce, tso, tco, rs, u, cscale);
                }
            }
            const unsigned int lad = coefs + (CPL ? QO_LAD_CPL : 0) * (unsigned int)sizeof(T);
#pragma unroll
            for (int e = 0; e < N; e++) {
                const bool series = ((e + FIRST) & 1) == 0;
                const unsigned int cf = lad + e * QO_LAD_STRIDE * (unsigned int)sizeof(T);
                if (series) {
                    if (e == 0 && !CPL) lad_ser_lossy_l<T, PTS, NROWS, true>(cf, w, w2, rs, u);
                    else lad_ser_lossy_l<T, PTS, NROWS, false>(cf, w, w2, rs, u);
                } else {
                    if (e == 0 && !CPL) lad_shunt_lossy_c<T, PTS, NROWS, true>(cf, w, wi, rs, u);
                    else lad_shunt_lossy_c<T, PTS, NROWS, false>(cf, w, wi, rs, u);
                }
            }
            const T rl = T(P.rl);
            T den2[PTS], s11m[PTS];
            QO_PTS {
                const T den_r = qfma(u.ar[0][p], rl, u.br[0][p]), den_i = qfma(u.ai[0][p], rl, u.bi[0][p]);
                den2[p] = qfma(den_r, den_r, den_i * den_i);
            }
            if (NROWS == 2) {
                /* |S11|^2 = |v . [Rl 1]|^2 / |den|^2 (the coupler's common factor 1/k cancels in the ratio) */
                T rd[PTS];
                lad_rcp_batch<PTS>(den2, rd);
                QO_PTS {
                    const T n_r = qfma(u.ar[1][p], rl, u.br[1][p]), n_i = qfma(u.ai[1][p], rl, u.bi[1][p]);
                    s11m[p] = qfma(n_r, n_r, n_i * n_i) * rd[p];
                }
            }
            if (CPL) { QO_PTS den2[p] *= cscale[p]; }
            /* Trackers.  Spec bands are contiguous in frequency, so nearly every warp-iteration sees ONE
             * mask value on all its points: a warp vote picks the fast path (a plain running max per active
             * spec, no per-point selects); iterations that straddle a band edge take the general path. */
            unsigned int m_or = mk[0], m_and = mk[0];
#pragma unroll
            for (int p = 1; p < PTS; p++) { m_or |= mk[p]; m_and &= mk[p]; }
            const unsigned int any = __reduce_or_sync(0xffffffffu, m_or), all = __reduce_and_sync(0xffffffffu, m_and);
            if (any == all) {
#pragma unroll
                for (int sp = 0; sp < QO_LAD_NSPEC; sp++) {
                    if ((all >> sp) & 1u) {
                        if (NROWS == 2 && P.is_s11[sp]) { QO_PTS trk[sp] = s11m[p] > trk[sp] ? s11m[p] : trk[sp]; }
                        else if (P.neg[sp]) { QO_PTS { const T c = -den2[p]; trk[sp] = c > trk[sp] ? c : trk[sp]; } }
                        else { QO_PTS trk[sp] = den2[p] > trk[sp] ? den2[p] : trk[sp]; }
                    }
                }
            } else {
#pragma unroll
                for (int sp = 0; sp < QO_LAD_NSPEC; sp++) {
                    if ((any >> sp) & 1u) {
                        QO_PTS {
                            const T val = (NROWS == 2 && P.is_s11[sp]) ? s11m[p] : (P.neg[sp] ? -den2[p] : den2[p]);
                            const T cand = ((mk[p] >> sp) & 1u) ? val : LadNum<T>::neg_huge();
                            trk[sp] = cand > trk[sp] ? cand : trk[sp];
                        }
                    }
                }
            }
        }

        /* 3. per-sample verdict: warp max of every tracker, then shared-memory counters */
        unsigned int fail = 0;
#pragma unroll
        for (int sp = 0; sp < QO_LAD_NSPEC; sp++) {
            if (sp < P.nspec) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    const T o = __shfl_xor_sync(0xffffffffu, trk[sp], off);
                    trk[sp] = o > trk[sp] ? o : trk[sp];
                }
                if ((double)trk[sp] > P.thr[sp]) fail |= 1u << sp;
            }
        }
        if (lane == 0) {
            qo_tally_one(s_cnt, P.nspec, fail);
            if (P.hist_spec >= 0) {
                double worst = 0.0;      /* |den|^2 (or |S11|^2) extreme of the histogram spec's band */
#pragma unroll
                for (int sp = 0; sp < QO_LAD_NSPEC; sp++) if (sp == P.hist_spec) worst = fabs((double)trk[sp]);
                const double k21 = P.k21;
                const double lin = P.hist_kind == SK_S11_MAX ? worst : P.hist_kind == SK_DEN2_MAX ? k21 * k21 / worst : k21 * k21 * (1.0 / worst);
                qo_tally_hist(s_cnt, P.nspec, qo_hist_bin(10.0 * log10(lin), P.hist_lo, P.hist_hi, P.hist_bins));
            }
        }
        s = __shfl_sync(0xffffffffu, s_next, 0);
    }
    __syncthreads();
    qo_tally_flush<TPB>(s_cnt, ncnt, P.counters);
}
