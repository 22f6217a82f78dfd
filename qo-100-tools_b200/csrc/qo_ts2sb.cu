/*
 * qo_ts2sb.cu -- instantiations of the thread-per-sample kernel's histogram-screen flavour (qo_ts.cuh::qo_mc_ts_screen_kernel) for plain
 * ladders, 6-8 numerator pairs (one translation unit per range, as qo_ts2a.cu ... qo_ts2c.cu: they compile in parallel).
 */
#include <cuda_runtime.h>
#include "qo_ts.cuh"
#include "qo_ts_launch.h"

extern "C" ts_fn qo_ts_screen_kernel_b(int kn)
{
    switch (kn) {
    case 6: return qo_mc_ts_screen_kernel<QO_TS_PT2, QO_TS_MINB2, 6>;
    case 7: return qo_mc_ts_screen_kernel<QO_TS_PT2, QO_TS_MINB2, 7>;
    case 8: return qo_mc_ts_screen_kernel<QO_TS_PT2, QO_TS_MINB2, 8>;
    default: return nullptr;
    }
}
