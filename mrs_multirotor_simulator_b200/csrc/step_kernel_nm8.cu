// step_kernel_nm8.cu — instantiates the stepping kernels for 8 motors (see step_kernel.cuh)
#include "step_kernel.cuh"

template void launch_step_nm<8>(const DevState&, const DevParams*, uint32_t*, double, int, int, bool, cudaStream_t, int*);
