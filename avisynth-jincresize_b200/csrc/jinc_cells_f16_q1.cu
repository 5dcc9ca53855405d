// piecewise-periodic rational-ratio kernels, source step 1 per cell, for half (IEEE binary16) planes, staged as float
#include "jinc_cells.cuh"

namespace jinc_rs {
template int launch_cells_q<__half, 1>(const jinc_table*, CellsArgs&, int, cudaStream_t, const Rect*, int);
}
