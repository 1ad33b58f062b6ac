// abi_internal.h -- shared between abi.cu (the stateless entry points) and host_env.cu (the host-buffer front end).
#pragma once
#include "launch.h"
#include "tick_core.cuh"

namespace tron {

inline size_t align256(size_t x) { return (x + 255u) & ~(size_t)255u; }
inline bool geometry_ok(int n, int w, int h) { return n > 0 && w >= 2 && h >= 2 && w <= 126 && h <= 126; }
inline int planes_of(int enc) { return enc == TRON_ENC_LUT1 ? 1 : enc == TRON_ENC_POPUP3 ? 3 : enc == TRON_ENC_POPUP3_CONST ? 4 : 0; }
inline int enc_kind_of(int enc) { return enc == TRON_ENC_LUT1 ? 1 : enc == TRON_ENC_POPUP3 ? 2 : enc == TRON_ENC_POPUP3_CONST ? 3 : 0; }
// layouts whose state is a set of dense arrays over all games (a chunk of games is addressed by StepParams::state_off)
inline bool layout_is_dense(int layout) { return layout == TRON_LAYOUT_TRAIL || layout == TRON_LAYOUT_BITS; }

// bytes of grid state per game (TRAIL / BITS: summed over their dense arrays)
size_t grid_stride(int layout, int w, int h);
// kernel parameters from the public argument block (mode: MODE_STEP | MODE_OBSERVE | MODE_RESET)
int fill_params(const tron_step_args* a, int mode, StepParams& p);
// narrow a whole-batch parameter block to the games [lo, lo+n)
void slice_params(const StepParams& base, int lo, int n, StepParams& p);
int dispatch(const StepParams& p, int mode, int obs_dtype, int obs_enc, cudaStream_t s);

// RAII: run a call on a given device, restore the caller's device afterwards
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; prev = -1; return; }
        if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess; else prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace tron
