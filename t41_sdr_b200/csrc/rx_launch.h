/* rx_launch.h — launchers of the kernels that live in units of their own (the throughput kernel, rx_fast.cu; the rows-only
   kernel, rx_rows.cu), called from the C-ABI (rx_api.cu). */
#ifndef T41RX_LAUNCH_H
#define T41RX_LAUNCH_H

#include <cuda_runtime.h>

namespace t41rx {

struct LaunchArgs;

cudaError_t ConfigureStreamKernel();
cudaError_t LaunchStreamKernel(const LaunchArgs &a, int n_sms, cudaStream_t st);
int StreamKernelMaxReceiversPerCta();

cudaError_t ConfigureRowsKernel();
cudaError_t LaunchRowsKernel(const LaunchArgs &a, int n_sms, cudaStream_t st);
long long RowsDcRefilterCount();                                        /* < 0: error */
cudaError_t RowsPhaseCycles(unsigned long long *out64, int reset);     /* developer builds (T41RX_PHASE_TIMING) */

/* entry points in other units (the channelizer, rx_chan.cu) report failures through t41rx_last_error(): sets its text
   on the calling thread and returns code */
int SetApiError(int code, const char *text);

}  // namespace t41rx
#endif
