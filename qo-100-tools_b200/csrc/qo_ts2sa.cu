/*
 * qo_ts2sa.cu -- instantiations of the thread-per-sample kernel's histogram-screen flavour (qo_ts.cuh::qo_mc_ts_screen_kernel) for plain
 * ladders, 2-5 numerator pairs (one translation unit per range, as qo_ts2a.cu ... qo_ts2c.cu: they compile in parallel).
 */
#include <cuda_runtime.h>
#include "qo_ts.cuh"
#include "qo_ts_launch.h"

extern "C" ts_fn qo_ts_screen_kernel_a(int kn)
{
    switch (kn) {
    case 2: return qo_mc_ts_screen_kernel<QO_TS_PT2, QO_TS_MINB2, 2>;
    case 3: return qo_mc_ts_screen_kernel<QO_TS_PT2, QO_TS_MINB2, 3>;
    case 4: return qo_mc_ts_screen_kernel<QO_TS_PT2, QO_TS_MINB2, 4>;
    case 5: return qo_mc_ts_screen_kernel<QO_TS_PT2, QO_TS_MINB2, 5>;
    default: return nullptr;
    }
}
