/*
 * qo_spot.cuh -- spot-frequency Monte-Carlo kernel (sm_100a, FP64): yield at a HANDFUL of frequencies per sample.
 *
 * BASELINE config 3 ("PA LPF ... harmonic-rejection yield at 2.4/4.8/7.2 GHz, 1e7 samples"; reference markers
 * util/pa-lpf-simulation/pa-lpf-simulation.dpl:25-27) evaluates 3 points per sample.  The warp-per-sample kernels
 * (qo_tf.cuh, qo_ladder.cuh, qo_lumped.cuh) spread one sample's grid over 32 lanes, so with <= 8 points most lanes idle
 * and the per-sample work (variates, element records) is paid at 1/32 lane efficiency.  Here ONE THREAD owns one sample:
 * it draws its variates (one Philox block per two variables, bit-exact twin of the C stream), walks the lumped
 * branches once, and carries the row vectors u = [1 Rs] M1...Mk (and v = [1 -Rs] M1...Mk for |S11| specs) of ALL its
 * points in registers -- series Z: b += a Z, shunt Y: a += b Y, with Z = N(jw)/D(jw) from the rational branch table of
 * qo_tf_core.h.  Specs are compared per point in linear power; pass / per-spec fail counts go through warp ballots,
 * the histogram through shared-memory atomics, one global atomic per counter per block at the end.
 */
#pragma once
#include "qo_lumped.cuh"
#include "qo_tf_core.h"

#define QO_SPOT_MAXF 8           /* frequencies per sample kept in registers */
#define QO_SPOT_MAXEL 24
#define QO_SPOT_TPB 128

struct SpotParams {
    const DevProg *prog;
    unsigned long long *counters;
    unsigned long long sample_offset, nsamples, seed;
    double rs, rl, k21, hist_lo, hist_hi;
    double w[QO_SPOT_MAXF];                  /* angular frequencies */
    unsigned int mask[QO_SPOT_MAXF];         /* spec bits per point */
    double thr[QO_NSPEC_MAX];                /* canonical thresholds (DevProg::spec_thr) */
    int kind[QO_NSPEC_MAX];                  /* SK_DEN2_MAX | SK_DEN2_MIN | SK_S11_MAX */
    int nf, n_el, el0, nspec, dist, hist_spec, hist_bins;
};

template <bool S11>
__global__ void __launch_bounds__(QO_SPOT_TPB, 4) qo_mc_spot_kernel(const __grid_constant__ SpotParams P)
{
    constexpr int F = QO_SPOT_MAXF;
    __shared__ double s_nom[QO_SPOT_MAXEL][6], s_tol[QO_SPOT_MAXEL][6];
    __shared__ short s_var[QO_SPOT_MAXEL][6];
    __shared__ unsigned char s_mode[QO_SPOT_MAXEL][6];
    __shared__ int s_op[QO_SPOT_MAXEL];
    __shared__ unsigned int s_cnt[QO_NCNT_MAX];
    const int ncnt = qo_ncnt(P.nspec, P.hist_bins);
    qo_tally_zero<QO_SPOT_TPB>(s_cnt, ncnt);
    for (int i = threadIdx.x; i < P.n_el * 6; i += QO_SPOT_TPB) {
        const int e = i / 6, k = i - 6 * e;
        s_nom[e][k] = P.prog->nom[P.el0 + e][k]; s_tol[e][k] = P.prog->ttol[P.el0 + e][k];
        s_var[e][k] = P.prog->tvar[P.el0 + e][k]; s_mode[e][k] = P.prog->tmode[P.el0 + e][k];
    }
    for (int i = threadIdx.x; i < P.n_el; i += QO_SPOT_TPB) s_op[i] = P.prog->opcode[P.el0 + i];
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int nf = P.nf;
    const double rs = P.rs, rl = P.rl;
    const unsigned long long stride = (unsigned long long)gridDim.x * QO_SPOT_TPB;
    /* warp-uniform trip count: the ballots below are full-warp collectives */
    for (unsigned long long base = (unsigned long long)blockIdx.x * QO_SPOT_TPB + (threadIdx.x & ~31u); base < P.nsamples; base += stride) {
        const unsigned long long s = base + lane;
        const bool valid = s < P.nsamples;
        unsigned int fail = 0;
        double worst = 0.0;
        bool have_worst = false;
        if (valid) {
            double ar[F], ai[F], br[F], bi[F], cr[F], ci[F], dr_[F], di_[F];      /* u = (a, b); v = (c, d) for |S11| */
#pragma unroll
            for (int t = 0; t < F; t++) { ar[t] = 1.0; ai[t] = 0.0; br[t] = rs; bi[t] = 0.0; cr[t] = 1.0; ci[t] = 0.0; dr_[t] = -rs; di_[t] = 0.0; }
            unsigned int blk = 0xffffffffu;
            uint32_t c4[4] = { 0, 0, 0, 0 };
            for (int e = 0; e < P.n_el; e++) {
                double p[6];
#pragma unroll
                for (int k = 0; k < 6; k++) {
                    p[k] = s_nom[e][k];
                    const int tv = s_var[e][k];
                    if (tv >= 0) {
                        /* one Philox block serves variables 2b and 2b+1 (qo_stream.h contract) */
                        if ((unsigned int)(tv >> 1) != blk) {
                            blk = (unsigned int)(tv >> 1);
                            const unsigned long long gs = P.sample_offset + s;
                            c4[0] = (uint32_t)gs; c4[1] = (uint32_t)(gs >> 32); c4[2] = blk; c4[3] = 0u;
                            qo_philox_rounds(c4, (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
                        }
                        const uint64_t wbits = (tv & 1) ? (((uint64_t)c4[3] << 32) | c4[2]) : (((uint64_t)c4[1] << 32) | c4[0]);
                        p[k] = qo_stream_apply(p[k], s_tol[e][k], qo_stream_from_bits53(wbits >> 11, P.dist), s_mode[e][k]);
                    }
                }
                double nd[6];
                const int series = qo_tf_element(s_op[e], p, 1.0, nd);
#pragma unroll
                for (int t = 0; t < F; t++) {
                    if (t < nf) {
                        const double w = P.w[t], y = -w * w;
                        const double nr = fma(nd[2], y, nd[0]), ni = nd[1] * w, dr = fma(nd[5], y, nd[3]), di = nd[4] * w;
                        const double inv = qrcp(fma(dr, dr, di * di));
                        const double zr = fma(nr, dr, ni * di) * inv, zi = fma(ni, dr, -nr * di) * inv;
                        if (series) {
                            br[t] = fma(ar[t], zr, fma(-ai[t], zi, br[t])); bi[t] = fma(ar[t], zi, fma(ai[t], zr, bi[t]));
                            if (S11) { dr_[t] = fma(cr[t], zr, fma(-ci[t], zi, dr_[t])); di_[t] = fma(cr[t], zi, fma(ci[t], zr, di_[t])); }
                        } else {
                            ar[t] = fma(br[t], zr, fma(-bi[t], zi, ar[t])); ai[t] = fma(br[t], zi, fma(bi[t], zr, ai[t]));
                            if (S11) { cr[t] = fma(dr_[t], zr, fma(-di_[t], zi, cr[t])); ci[t] = fma(dr_[t], zi, fma(di_[t], zr, ci[t])); }
                        }
                    }
                }
            }
#pragma unroll
            for (int t = 0; t < F; t++) {
                if (t < nf) {
                    const double er = fma(ar[t], rl, br[t]), ei = fma(ai[t], rl, bi[t]);
                    const double den2 = fma(er, er, ei * ei);
                    double s11v = 0.0;
                    if (S11) {
                        const double fr = fma(cr[t], rl, dr_[t]), fi = fma(ci[t], rl, di_[t]);
                        s11v = fma(fr, fr, fi * fi) / den2;
                    }
                    const unsigned int mb = P.mask[t];
                    for (int sp = 0; sp < P.nspec; sp++) {
                        if (!((mb >> sp) & 1u)) continue;
                        const int sk = P.kind[sp];
                        const double v = sk == SK_S11_MAX ? s11v : den2;
                        const bool bad = sk == SK_DEN2_MIN ? (v < P.thr[sp]) : (v > P.thr[sp]);
                        if (bad) fail |= 1u << sp;
                        if (sp == P.hist_spec) {
                            const bool better = sk == SK_DEN2_MIN ? (v < worst) : (v > worst);
                            if (!have_worst || better) { worst = v; have_worst = true; }
                        }
                    }
                }
            }
        }
        qo_tally_warp(s_cnt, P.nspec, fail, __ballot_sync(0xffffffffu, valid));
        if (valid && P.hist_spec >= 0) {
            const int sk = P.kind[P.hist_spec];
            const double k21 = P.k21;
            const double lin = sk == SK_S11_MAX ? worst : sk == SK_DEN2_MAX ? k21 * k21 / worst : k21 * k21 * (1.0 / worst);
            qo_tally_hist(s_cnt, P.nspec, qo_hist_bin(10.0 * log10(lin), P.hist_lo, P.hist_hi, P.hist_bins));
        }
    }
    __syncthreads();
    qo_tally_flush<QO_SPOT_TPB>(s_cnt, ncnt, P.counters);
}
