// integer-ratio downscale kernels for half (IEEE binary16) planes: float pairs and tiles, as for float planes
#include "jinc_down.cuh"

namespace jinc_rs {
template int launch_down<__half>(const jinc_table*, DownArgs&, int, const int*, bool, int, cudaStream_t, const Rect*, int);
}
