// snk_grid_class.cuh -- the class of a SNK_OBS_GRID cell code in view `view` (the order of SNK_GRID_CONV_CLASSES in
// include/snk.h), shared by the first-layer kernels of snk_grid_conv.cu and snk_grid_conv84.cu.
#pragma once
#include "../../include/snk.h"

// code 2 is unused and drawn black
static __device__ __forceinline__ unsigned cell_class(unsigned c, int view) {
  if (c == SNK_CELL_WALL) return 2u;
  if (c < 3u) return c == SNK_CELL_FRUIT ? 1u : 0u;
  return (((c - 3u) >> 1) == (unsigned)view ? 3u : 5u) + ((c - 3u) & 1u);
}
