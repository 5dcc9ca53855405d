// exact-2x interior kernels for half (IEEE binary16) planes: float tiles, every tap multiplied
#include "jinc_up2x.cuh"

namespace jinc_rs {
template int launch_up2x<__half>(const jinc_table*, UpArgs&, long long, int, cudaStream_t);
}
