// step_c144.cu -- fused tick kernels specialised for the reference's config.py grid (10x10 -> 144 cells).
#include "step_dispatch.cuh"

namespace tron {
// games per CTA for the 144-cell kernels: 128 (one per thread) when there are enough games to fill the GPU, fewer for small batches
int tile_envs_small_grid(int n_envs) {
    // one wave of CTAs if the batch allows it: 8 CTAs are resident per SM, so ceil(n / (8 * SMs)) games per CTA (a multiple of 16)
    // puts every game on the machine at once (65,536 games -> 64 per CTA -> 1024 CTAs <= 1184 slots); big batches use 128.
    const int slots = 8 * sm_count();
    int g = (n_envs + slots - 1) / slots;
    g = (g + 15) & ~15;
    return g < 16 ? 16 : (g > 128 ? 128 : g);
}
int launch_step_c144(const StepParams& p_in, int mode, int obs_dtype, int enc_kind, cudaStream_t s) {
    StepParams p = p_in;
    p.G = tile_envs_small_grid(p.N);
    return launch_mode<144, 8>(p, mode, obs_dtype, enc_kind, s);
}
}  // namespace tron
