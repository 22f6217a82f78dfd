/*
 * qo_nodal_prog.h -- the device-side description of a nodal job (SURVEY row N4; reference network
 * util/pa-bias-simulation/pa-bias-simulation.sch:19-72) and the per-sample verdict.  Shared, as text, between the
 * ahead-of-time kernels of qo_nodal.cu and the run-time compiled kernel (qo_nodal_jit.h hands this file to NVRTC), so it
 * includes nothing: the includer provides the fixed-width integer types, QO_NODAL_MAX_BR / QO_NODAL_MAX_PORTS and qo_tally.cuh.
 */
#ifndef QO_NODAL_PROG_H
#define QO_NODAL_PROG_H
#define QN_TPB 64
#define QN_MAX_SPEC 8
#define QN_MAX_VAR 64

struct NodalProg {
    int32_t n_nodes, nb, np, n_unk, nspec, hist_spec, hist_bins, n_var, dist, full;
    uint64_t seed;
    double hist_lo, hist_hi;
    int32_t port_node[QO_NODAL_MAX_PORTS];
    double port_z0[QO_NODAL_MAX_PORTS];
    int32_t kind[QO_NODAL_MAX_BR];
    int32_t node[QO_NODAL_MAX_BR][4];
    double nom[QO_NODAL_MAX_BR][4];
    double ttol[QO_NODAL_MAX_BR][4];
    int16_t tvar[QO_NODAL_MAX_BR][4];
    uint8_t tmode[QO_NODAL_MAX_BR][4];
    int32_t spec_min[QN_MAX_SPEC], spec_row[QN_MAX_SPEC], spec_col[QN_MAX_SPEC];   /* spec_min: 1 = "|S| >= limit" */
    double spec_thr[QN_MAX_SPEC];       /* linear |S|^2 threshold */
    double spec_limit_db[QN_MAX_SPEC];
};

/* one sample's verdict, once the block has walked its points: the block maximum of every spec's tracker (trk[sp]: the thread's
 * running maximum of |S|^2, negated for "|S| >= limit" specs, -1e300 where the spec covered none of its points) against the
 * threshold, then thread 0 tallies the sample.  Called by every thread of the block; N >= nspec */
template <int N>
__device__ __forceinline__ void qn_verdict(const NodalProg *prog, int nspec, const double (&trk)[N], double (*s_trk)[QN_TPB / 32],
                                           unsigned int *s_cnt)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int sp = 0; sp < N; sp++) {
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
        qo_tally_one(s_cnt, nspec, fail);
        if (prog->hist_bins > 0) qo_tally_hist(s_cnt, nspec, qo_hist_bin(10.0 * log10(hist_worst), prog->hist_lo, prog->hist_hi, prog->hist_bins));
    }
}
#endif
