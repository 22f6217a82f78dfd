/*
 * qo_ts.cu -- instantiations and launcher of the thread-per-sample transfer-function kernel (qo_ts.cuh).
 * The kernels themselves are instantiated in qo_ts2a.cu, qo_ts2b.cu, qo_ts2c.cu, qo_ts4.cu and, behind the histogram screen,
 * qo_ts2sa.cu ... qo_ts2sc.cu (most of the library's compile time, hence in parallel).  Development builds:
 * -DQO_TS_DEV_KN=9 -DQO_TS_DEV_KE=14 -DQO_TS_DEV_KN2=8 -DQO_TS_DEV_KE2=8 compiles those loop bodies only.
 */
#include <cuda_runtime.h>
#include "qo_ts.cuh"
#include "qo_tf_launch.h"
#include "qo_ts_launch.h"

/* ---- thread-per-sample flavour (qo_ts.cuh) ------------------------------------------------------------------- */
/* Can the bulk of this plan's launches run thread-per-sample?  Plain |S21| jobs with at most four specs whose kept polynomial
 * lengths fit the register capacities; behind a coupler only the matched / uniform-grid / equal-angle form (config 5). */
extern "C" int qo_ts_eligible(const TfPlan *tp, int nspec, int cpl_rot_same)
{
    if (tp->s11 || tp->gd || nspec > 4) return 0;
    if (tp->den != QO_TF_DEN_NONE && tp->den != QO_TF_DEN_E) return 0;
    if (tp->kn < 2 || (tp->den == QO_TF_DEN_E && (tp->kd < 2 || (tp->kd & 1)))) return 0;
    if (tp->cpl_op < 0) return tp->nn == 2 && tp->kn <= QO_TS_CAPN2 && (tp->den == QO_TF_DEN_NONE || tp->kd <= QO_TS_CAPE2);
    return cpl_rot_same && tp->nn == 4 && tp->kn <= QO_TS_CAPN4 && (tp->den == QO_TF_DEN_NONE || tp->kd <= QO_TS_CAPE4);
}

static ts_fn ts_pick_kernel(const TfPlan *tp)
{
    if (tp->cpl_op >= 0) return qo_ts_kernel_4(tp->kn);
    if (tp->ts_nseed > 0)                /* the plan screens the histogram band (tf_hist_screen) */
        return tp->kn <= 5 ? qo_ts_screen_kernel_a(tp->kn) : tp->kn <= 8 ? qo_ts_screen_kernel_b(tp->kn) : qo_ts_screen_kernel_c(tp->kn);
    return tp->kn <= 5 ? qo_ts_kernel_2a(tp->kn) : tp->kn <= 8 ? qo_ts_kernel_2b(tp->kn) : qo_ts_kernel_2c(tp->kn);
}

/* blocks of this plan's kernel that are resident on one SM at the same time (what the hardware grants, not what
 * __launch_bounds__ asked for): the grid is exactly one wave of them, so that the static deal of samples is balanced */
static int ts_blocks_per_sm(const TfPlan *tp)
{
    int occ = 0;
    ts_fn fn = ts_pick_kernel(tp);
    if (!fn || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, QO_TS_TPB, 0) != cudaSuccess) { cudaGetLastError(); occ = 0; }
    return occ;
}

/* points per group of this plan's kernel (the launcher builds the run table in groups) */
extern "C" int qo_ts_group_points(const TfPlan *tp) { return tp->cpl_op < 0 ? QO_TS_PT2 : QO_TS_PT4; }

/* threads of one full wave of the thread-per-sample kernel */
extern "C" int qo_ts_wave_threads(const TfPlan *tp, int sm_count) { return sm_count * ts_blocks_per_sm(tp) * QO_TS_TPB; }

extern "C" int qo_ts_launch(const TfPlan *tp, int sm_count, const TsParams *Q, cudaStream_t st)
{
    const int bps = ts_blocks_per_sm(tp);
    if (bps <= 0) return (int)cudaErrorLaunchOutOfResources;
    ts_pick_kernel(tp)<<<(unsigned)(sm_count * bps), QO_TS_TPB, 0, st>>>(*Q);
    return (int)cudaGetLastError();
}

