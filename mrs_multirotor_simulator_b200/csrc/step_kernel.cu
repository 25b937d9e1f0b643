// step_kernel.cu — dispatch of the stepping kernels (step_kernel.cuh, instantiated per motor count in
// step_kernel_nm*.cu) plus the small kernels around them: position publishing and the per-launch
// parameter preparation.
#include <cstdlib>

#include "internal.h"

template <int NM_T>
void launch_step_nm(const DevState& s, const DevParams* uniform_params, uint32_t* sweep, double dt, int k_substeps, int uniform_mode, bool any_moment, cudaStream_t stream, int* info);

int launch_step(const DevState& s, const DevParams* uniform_params, uint32_t* sweep, double dt, int k_substeps, int uniform_mode, int uniform_nm, bool any_moment,
                cudaStream_t stream, int* info) {
  int scratch[4];
  if (!info) info = scratch;
  info[0] = info[1] = info[2] = info[3] = 0;
  if (s.n <= 0) return 0;
  switch (uniform_nm) {
    case 4:
      launch_step_nm<4>(s, uniform_params, sweep, dt, k_substeps, uniform_mode, any_moment, stream, info);
      break;
    case 6:
      launch_step_nm<6>(s, uniform_params, sweep, dt, k_substeps, uniform_mode, any_moment, stream, info);
      break;
    case 8:
      launch_step_nm<8>(s, uniform_params, sweep, dt, k_substeps, uniform_mode, any_moment, stream, info);
      break;
    default:
      launch_step_nm<0>(s, uniform_params, sweep, dt, k_substeps, uniform_mode, any_moment, stream, info);
      break;
  }
  return 1;
}

namespace {
__device__ __forceinline__ uint32_t fenc(float f) {
  const uint32_t b = __float_as_uint(f);
  return (b >> 31) ? ~b : (b | 0x80000000u);
}

// positions of the state -> packed buffer (after set_state / a parity flip), plus the per-warp bounding boxes the peers filter by
__global__ void __launch_bounds__(256) publish_positions_kernel(DevState s) {
  const int64_t i      = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;  // external index; blockDim is a multiple of 32: warps coincide with the 32-UAV groups
  const bool    inside = i < s.n;
  double        x = 0.0, y = 0.0, z = 0.0;
  if (inside) {
    const int64_t slot = s.perm ? int64_t(s.perm[i]) : i;
    x          = s.st[tix(ST_ROWS, 0, slot)];
    y          = s.st[tix(ST_ROWS, 1, slot)];
    z          = s.st[tix(ST_ROWS, 2, slot)];
    double* gp = s.gpos + 3 * (s.shard_begin + i);
    gp[0]      = x;
    gp[1]      = y;
    gp[2]      = z;
  }
  if (s.gbox) {
    const uint32_t full = 0xffffffffu;
    uint32_t lo0 = inside ? fenc(__double2float_rd(x)) : 0xFFFFFFFFu, lo1 = inside ? fenc(__double2float_rd(y)) : 0xFFFFFFFFu,
             lo2 = inside ? fenc(__double2float_rd(z)) : 0xFFFFFFFFu;
    uint32_t hi0 = inside ? fenc(__double2float_ru(x)) : 0u, hi1 = inside ? fenc(__double2float_ru(y)) : 0u, hi2 = inside ? fenc(__double2float_ru(z)) : 0u;
    lo0 = __reduce_min_sync(full, lo0);
    lo1 = __reduce_min_sync(full, lo1);
    lo2 = __reduce_min_sync(full, lo2);
    hi0 = __reduce_max_sync(full, hi0);
    hi1 = __reduce_max_sync(full, hi1);
    hi2 = __reduce_max_sync(full, hi2);
    if ((threadIdx.x & 31) == 0 && i < s.n_groups32 * 32) {
      uint32_t* row = s.gbox + 6 * (i >> 5);
      row[0] = lo0, row[1] = lo1, row[2] = lo2, row[3] = hi0, row[4] = hi1, row[5] = hi2;
    }
  }
}

// exp(-dt / tau) (MM:244) once per parameter set, on the device: every stepping-kernel variant reads the same bits
__global__ void prep_params_kernel(DevParams* params, int n_sets, double dt) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n_sets) params[k].filt = exp(dt * params[k].neg_inv_tau);
}
}  // namespace

int launch_prep_params(DevParams* params, int n_sets, double dt, cudaStream_t stream) {
  if (n_sets <= 0) return 0;
  prep_params_kernel<<<(n_sets + 127) / 128, 128, 0, stream>>>(params, n_sets, dt);
  return 1;
}

int launch_publish_positions(const DevState& s, cudaStream_t stream) {
  if (s.n <= 0) return 0;
  publish_positions_kernel<<<unsigned((s.n + 255) / 256), 256, 0, stream>>>(s);
  return 1;
}
