// step_dispatch.cuh -- host side of the fused kernels: the one table that turns a run-time call into kernel template arguments, the
// shared-memory residency cap, and the launcher of step_tile_kernel for one geometry class.
#pragma once
#include <type_traits>

#include "launch.h"
#include "step_kernels.cuh"

namespace tron {

template <int V>
using Int = std::integral_constant<int, V>;

// The instantiations of a fused kernel: (mode, obs dtype, enc_kind) -> launch(Int<MODE>, Int<OD>, Int<LP>, std::bool_constant<CP>), with
// LP lut planes and CP the const plane (enc_kind 1: LP 1; 2: LP 3; 3: LP 3 + CP).  A reset, and a step without observations, use
// <MODE, TRON_I8, 0, false>.  Anything else without a kernel (an observation without planes, an unknown dtype) is TRON_ERR_INVALID.
template <class F>
int dispatch_obs(int mode, int od, int enc_kind, F&& launch) {
    if (mode == MODE_RESET) return launch(Int<MODE_RESET>(), Int<TRON_I8>(), Int<0>(), std::false_type());
    if (mode == MODE_STEP && enc_kind == 0) return launch(Int<MODE_STEP>(), Int<TRON_I8>(), Int<0>(), std::false_type());
    const auto with_enc = [&](auto mode_c, auto od_c) -> int {
        switch (enc_kind) {
            case 1: return launch(mode_c, od_c, Int<1>(), std::false_type());
            case 2: return launch(mode_c, od_c, Int<3>(), std::false_type());
            case 3: return launch(mode_c, od_c, Int<3>(), std::true_type());
            default: return TRON_ERR_INVALID;
        }
    };
    const auto with_dtype = [&](auto mode_c) -> int {
        if (od == TRON_BF16) return with_enc(mode_c, Int<TRON_BF16>());
        if (od == TRON_F32) return with_enc(mode_c, Int<TRON_F32>());
        if (od == TRON_I8) return with_enc(mode_c, Int<TRON_I8>());
        return TRON_ERR_INVALID;
    };
    if (mode == MODE_STEP) return with_dtype(Int<MODE_STEP>());
    if (mode == MODE_OBSERVE) return with_dtype(Int<MODE_OBSERVE>());
    return TRON_ERR_INVALID;
}

// Cells per encode item of a kernel whose other dtypes use CH.  f32 planes take at most 4, so that one warp-wide STG.128 covers whole
// 32-byte sectors (8 cells would give each lane two half-sector stores; measured 78% -> see profiles/r1_step_f32_lut1_2M.json).
constexpr int obs_ch(int od, int ch) { return od == TRON_F32 && ch == 8 ? 4 : ch; }

// Dynamic shared memory that caps the resident CTAs per SM at `cap`: floor(228 KB / (smem + 1 KB reserved)) == cap.  The fused kernels
// are write streams; with fewer of them per SM than the register limit allows, the DRAM pages see longer bursts.  Returns `smem`
// unchanged when it already allows fewer CTAs, or when the padding would exceed 200 KB.
inline size_t smem_for_ctas_per_sm(size_t smem, long long cap) {
    const size_t want = (size_t)(228 * 1024) / (size_t)(cap + 1) - 1024 + 256;
    return want > smem && want <= 200 * 1024 ? want : smem;
}

constexpr int kThreads = 128;
extern long long g_tile_ctas_per_sm;  // TRON_OPT_TILE_CTAS_PER_SM (abi.cu)
// measured defaults (profiles/r2_cta_cap_sweep.jsonl): 5 at 10x10 (+1.5-2 %), 6 for >= 2048 cells (+2 %), no cap in between (8x8, 32x32 lose)
inline long long default_tile_ctas(int C) { return C == 144 ? 5 : C >= 2048 ? 6 : 32; }

inline size_t tile_smem_bytes(int G, int C) {
    return (size_t)((G * C + 15) & ~15) + (size_t)((C + 15) & ~15) + (size_t)G * 4 + (size_t)G + 8 + 16 + 16 + 6 * sizeof(PlaneTab);
}

template <int C_T, int OD, int LP, bool CP, int CH, int MODE>
int launch_one(const StepParams& p, cudaStream_t s) {
    auto kern = step_tile_kernel<C_T, kThreads, OD, LP, CP, CH, MODE>;
    size_t smem = tile_smem_bytes(p.G, p.C);
    const unsigned grid = (unsigned)(((long long)p.N + p.G - 1) / p.G);
    const long long cap = g_tile_ctas_per_sm > 0 ? g_tile_ctas_per_sm : default_tile_ctas(p.C);
    if (LP > 0 && MODE == MODE_STEP && cap < 32 && grid > 8u * (unsigned)sm_count()) smem = smem_for_ctas_per_sm(smem, cap);
    if (smem > 48 * 1024 && ensure_dynamic_smem((const void*)kern, smem) != TRON_OK) return TRON_ERR_CUDA;
    kern<<<grid, kThreads, smem, s>>>(p);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

// p.G (games per CTA) is set by the caller
template <int C_T, int CH>
int launch_mode(const StepParams& p, int mode, int od, int enc_kind, cudaStream_t s) {
    return dispatch_obs(mode, od, enc_kind, [&](auto mode_c, auto od_c, auto lp, auto cp) {
        return launch_one<C_T, od_c, lp, cp, obs_ch(od_c, CH), mode_c>(p, s);
    });
}

}  // namespace tron
