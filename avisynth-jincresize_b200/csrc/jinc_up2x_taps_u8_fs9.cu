// exact-2x interior kernels of uint8_t planes, fs 9, with the zero taps of a tap-mask variant skipped
#include "jinc_up2x.cuh"

namespace jinc_rs {
template int launch_up2x_taps<uint8_t, 9>(const jinc_table*, UpArgs&, long long, int, cudaStream_t);
}
