// Langevin kernels for dim > 64 (langevin_wide.cu), reached from tsu_langevin_run.
#pragma once
#include <stdint.h>

#include "langevin_body.cuh"

namespace tsu_langevin {

// Caps of the wide kernels.  The Philox counter carries the block index b = i / PER in 16 bits, so no chain can
// draw more than 65536 blocks: 131072 coordinates in float64 (2 normals a block), 262144 in float32 (4 a block).
// QUADRATIC_FORM keeps a tile of chains in shared memory (64 bytes per coordinate), which bounds it at 2048;
// MIXTURE takes at most 16 centres.
constexpr int kWideMaxDimF64 = 131072;
constexpr int kWideMaxDimF32 = 262144;
constexpr int kWideMaxDimQForm = 2048;
constexpr int kWideMaxCentres = 16;

// dtype 0 = float32, 1 = float64; mixture_k = number of centres (MIXTURE only)
int langevin_wide_launch(const LangevinParams& P, int dtype, int mixture_k, uintptr_t stream);

}  // namespace tsu_langevin
