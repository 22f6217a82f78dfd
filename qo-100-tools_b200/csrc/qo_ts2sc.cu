/*
 * qo_ts2sc.cu -- instantiations of the thread-per-sample kernel's histogram-screen flavour (qo_ts.cuh::qo_mc_ts_screen_kernel) for plain
 * ladders, 9-10 numerator pairs (one translation unit per range, as qo_ts2a.cu ... qo_ts2c.cu: they compile in parallel).
 */
#include <cuda_runtime.h>
#include "qo_ts.cuh"
#include "qo_ts_launch.h"

extern "C" ts_fn qo_ts_screen_kernel_c(int kn)
{
    switch (kn) {
    case 9: return qo_mc_ts_screen_kernel<QO_TS_PT2, QO_TS_MINB2, 9>;
    case 10: return qo_mc_ts_screen_kernel<QO_TS_PT2, QO_TS_MINB2, 10>;
    default: return nullptr;
    }
}
