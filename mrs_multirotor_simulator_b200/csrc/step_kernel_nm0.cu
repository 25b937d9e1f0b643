// step_kernel_nm0.cu — instantiates the stepping kernels for a per-UAV motor count (see step_kernel.cuh)
#include "step_kernel.cuh"

template void launch_step_nm<0>(const DevState&, const DevParams*, uint32_t*, double, int, int, bool, cudaStream_t, int*);
