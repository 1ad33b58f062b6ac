// step_generic.cu -- fused tick kernels for any grid size (cells per env known only at run time).
#include "step_dispatch.cuh"

namespace tron {
// games per CTA: as many as fit ~18 KB of shared memory, at most one per thread, rounded so that a
// full tile is a multiple of 16 bytes (keeps the bulk-copy path usable).
long long g_tile_bytes = 18432;  // TRON_OPT_TILE_BYTES; measured best on B200 for 32x32 and 64x64 (more CTAs in flight beats bigger tiles)
static int tile_envs_generic(int cells) {
    int g = (int)(g_tile_bytes / cells);
    if (g > kThreads) g = kThreads;
    if (g < 1) g = 1;
    const int need = (cells % 16 == 0) ? 1 : (cells % 8 == 0) ? 2 : (cells % 4 == 0) ? 4 : (cells % 2 == 0) ? 8 : 16;
    if (g >= need) g -= g % need;
    return g;
}
int launch_step_generic(const StepParams& p_in, int mode, int obs_dtype, int enc_kind, cudaStream_t s) {
    StepParams p = p_in;
    p.G = tile_envs_generic(p.C);
    if (p.C % 4 == 0) return launch_mode<0, 4>(p, mode, obs_dtype, enc_kind, s);
    return launch_mode<0, 1>(p, mode, obs_dtype, enc_kind, s);
}
}  // namespace tron
