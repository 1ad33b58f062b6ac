// launch.h -- host-side launch entry points of the kernel translation units (internal, not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tron_b200.h"

namespace tron {

struct StepParams;

// SM count of the current device (cached per device; replaces the hard-coded 148)
int sm_count();
// opt a kernel into `bytes` of dynamic shared memory on the CURRENT device (the attribute is per device and per function;
// cached per (function, device), thread-safe)
int ensure_dynamic_smem(const void* kernel, size_t bytes);

__host__ __device__ inline int tron_elem(int dt) {
    return (dt == TRON_U8 || dt == TRON_I8) ? 1 : dt == TRON_BF16 ? 2 : dt == TRON_I64 ? 8 : 4;
}

// step_c144.cu (10x10 grids, compile-time geometry) and step_generic.cu (any W,H)
// enc_kind: 0 none, 1 = 1 lut plane, 2 = 3 lut planes, 3 = 3 lut planes + const plane
// The fused-kernel launchers choose the games per CTA (p.G) themselves.
int launch_step_c144(const StepParams& p, int mode, int obs_dtype, int enc_kind, cudaStream_t s);
int launch_step_generic(const StepParams& p, int mode, int obs_dtype, int enc_kind, cudaStream_t s);
int launch_step_sparse(const StepParams& p, cudaStream_t s);
int launch_step_trail(const StepParams& p, int mode, int obs_dtype, int enc_kind, cudaStream_t s);
size_t trail_game_bytes_host(int W, int H);
// export / import take a StepParams with geometry, layout, grid, state_off, state_N and N filled in
int launch_trail_export(const StepParams& p, int8_t* tiles, int8_t* heads, uint8_t* alive, uint8_t* done, uint8_t* winner, int32_t* ep_len, cudaStream_t s);
int launch_trail_import(const StepParams& p, const int8_t* tiles, const int8_t* heads, const uint8_t* alive, const uint8_t* done, const uint8_t* winner,
                        const int32_t* ep_len, cudaStream_t s);
int launch_step_bits10(const StepParams& p, int mode, int obs_dtype, int enc_kind, cudaStream_t s);
int launch_step_bits(const StepParams& p, int mode, int obs_dtype, int enc_kind, cudaStream_t s);
int launch_bits_export(const StepParams& p, const void* meta, int8_t* tiles, cudaStream_t s);
int launch_bits_import(const StepParams& p, const int8_t* tiles, bool derive_heads, cudaStream_t s);
int tile_envs_small_grid(int n_envs);

int launch_export_meta(const void* meta, int n, int8_t* heads, uint8_t* alive, uint8_t* done, uint8_t* winner, int32_t* ep_len, cudaStream_t s);
int launch_import_meta(void* meta, int n, int W, int H, const int8_t* heads, const uint8_t* alive, const uint8_t* done, const uint8_t* winner,
                       const int32_t* ep_len, const int8_t* tiles_for_heads, cudaStream_t s);
int launch_advance_counter(uint64_t* c, uint64_t delta, cudaStream_t s);
int launch_random_actions(uint8_t* actions, int n, uint64_t seed, uint64_t counter, const uint64_t* cdev, uint64_t base, cudaStream_t s);
int launch_select_actions(const void* q, int q_dtype, int n, float eps, uint8_t* actions, uint64_t seed, uint64_t counter, const uint64_t* cdev,
                          uint64_t base, cudaStream_t s);
int launch_minimax(const int8_t* tiles, int n, int W, int H, int player, int tie_mode, uint64_t seed, uint64_t counter, const uint64_t* cdev,
                   uint64_t base, uint8_t* actions, int32_t* values, int32_t* child_ties, cudaStream_t s);
int launch_pop_up(const void* obs, int in_dtype, int64_t n_maps, int cells, void* planes, int out_dtype, cudaStream_t s);
int launch_replay_push(const replay_ring* ring, uint64_t cursor, const void* s, const void* s2, const uint8_t* action, const float* reward,
                       const uint8_t* done, int done_stride, int64_t n, cudaStream_t st);
int launch_replay_gather(const replay_ring* ring, const int64_t* idx, int64_t k, void* out_s, void* out_s2, int out_dtype, int64_t* out_a,
                         float* out_r, float* out_d, cudaStream_t st);
int launch_replay_sample(int64_t size, int64_t k, uint64_t seed, uint64_t counter, int64_t* idx, cudaStream_t st);
int launch_replay_sample_gather(const replay_ring* ring, int64_t size, int64_t k, uint64_t seed, uint64_t counter, void* out_s, void* out_s2,
                                int out_dtype, int64_t* out_a, float* out_r, float* out_d, int64_t* out_idx, cudaStream_t st);
int launch_replay_frames_sample_gather(const replay_frames* fr, int64_t first_tick, int64_t n_ticks, int64_t k, uint64_t seed, uint64_t counter,
                                       void* out_s, void* out_s2, int out_dtype, int64_t* out_a, float* out_r, float* out_d, int64_t* out_idx,
                                       cudaStream_t st);
// state replay ring (step_bits.cu): the per-launch inputs besides the env's StepParams (validated by replay_states_sample_gather)
struct StateSample {
    const char* states;                   // [S, slot_bytes]
    long long slot_bytes, meta_off;       // meta_off: the tron_meta array's offset inside a slot
    const uint8_t* action;                // [S, N, 2]
    const unsigned long long* counter;    // [S] or NULL
    const int8_t* slide_params;           // [S, N, 4] or NULL
    long long first_tick, n_ticks, k;
    unsigned long long seed, counter_s;   // the sampler's key and counter
    int S, out_dtype, lp, env_i8;         // lp: lut planes (the const plane, if any, is plane lp); env_i8: the env's tables hold int8
    float const_val;                      // the const plane as the env's obs dtype stores it
    void *out_s, *out_s2;
    long long* out_a;
    float *out_r, *out_d;
    long long* out_idx;
};
int launch_replay_states(const StepParams& p, const StateSample& q, cudaStream_t s);
int debug_violations(uint64_t* count, int32_t* first_code);

}  // namespace tron
