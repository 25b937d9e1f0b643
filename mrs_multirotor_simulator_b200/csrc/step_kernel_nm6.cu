// step_kernel_nm6.cu — instantiates the stepping kernels for 6 motors (see step_kernel.cuh)
#include "step_kernel.cuh"

template void launch_step_nm<6>(const DevState&, const DevParams*, uint32_t*, double, int, int, bool, cudaStream_t, int*);
