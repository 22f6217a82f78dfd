/* qo_ts_launch.h -- the per-translation-unit kernel tables of the thread-per-sample kernel (qo_ts2a.cu ... qo_ts4.cu, qo_ts2sa.cu ... qo_ts2sc.cu) */
#pragma once
struct TsParams;
typedef void (*ts_fn)(const TsParams);
extern "C" ts_fn qo_ts_kernel_2a(int kn);      /* NN = 2, kn 2..5 */
extern "C" ts_fn qo_ts_kernel_2b(int kn);      /* NN = 2, kn 6..8 */
extern "C" ts_fn qo_ts_kernel_2c(int kn);      /* NN = 2, kn 9..10 */
extern "C" ts_fn qo_ts_kernel_4(int kn);       /* NN = 4 (coupled-line block in front), kn 2..8 */
extern "C" ts_fn qo_ts_screen_kernel_a(int kn);    /* NN = 2 behind the histogram screen (qo_ts2sa.cu ... qo_ts2sc.cu), kn 2..5 */
extern "C" ts_fn qo_ts_screen_kernel_b(int kn);    /* kn 6..8 */
extern "C" ts_fn qo_ts_screen_kernel_c(int kn);    /* kn 9..10 */
