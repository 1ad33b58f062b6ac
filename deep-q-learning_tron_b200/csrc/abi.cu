// abi.cu -- the extern "C" boundary declared in include/tron_b200.h: argument validation and kernel
// dispatch.  No torch types, no exceptions, no CPU fallback.  (Host-buffer front end: host_env.cu.)
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>

#include "abi_internal.h"

using namespace tron;

namespace tron {

long long g_sparse_min_cells = 1024;  // TRON_OPT_SPARSE_MIN_CELLS
long long g_encode_variant = 0;       // TRON_OPT_ENCODE_VARIANT
long long g_tile_ctas_per_sm = 0;    // TRON_OPT_TILE_CTAS_PER_SM
long long g_bits_ctas_per_sm = 0;    // TRON_OPT_BITS_CTAS_PER_SM (0 = the kernels' own default)
extern long long g_tile_bytes;

// ---- per-device facts ------------------------------------------------------------------------------
int sm_count() {
    static std::atomic<int> cache[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    int n = cache[dev].load(std::memory_order_relaxed);
    if (n == 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) { cudaGetLastError(); n = 148; }
        cache[dev].store(n, std::memory_order_relaxed);
    }
    return n;
}
int ensure_dynamic_smem(const void* kernel, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, size_t> limit;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return TRON_ERR_CUDA;
    std::lock_guard<std::mutex> lock(mu);
    size_t& cur = limit[std::make_pair(kernel, dev)];
    if (bytes > cur) {
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) { cudaGetLastError(); return TRON_ERR_CUDA; }
        cur = bytes;
    }
    return TRON_OK;
}

static inline bool layout_known(int layout) { return layout >= TRON_LAYOUT_TILE8 && layout <= TRON_LAYOUT_BITS; }
static inline bool layout_ok(int layout, int w, int h) {
    if (layout == TRON_LAYOUT_BITS10) return w == 10 && h == 10;
    if (layout == TRON_LAYOUT_BITS) return w * h <= 128;
    return true;
}
size_t grid_stride(int layout, int w, int h) {
    return layout == TRON_LAYOUT_BITS10 ? 32u : layout == TRON_LAYOUT_BITS ? 48u : layout == TRON_LAYOUT_TRAIL ? trail_game_bytes_host(w, h)
                                                                                                                : (size_t)(w + 2) * (size_t)(h + 2);
}

static uint16_t bf16_bits_of_int8(int v) {  // every int8 is exactly representable in bf16
    float f = (float)v;
    uint32_t u;
    memcpy(&u, &f, 4);
    return (uint16_t)(u >> 16);
}

// device lookup tables indexed by (tile & 7): WALL(-1) -> 7, EMPTY 0, bodies/heads/slides 1..6
static void build_device_tables(const int8_t lut6[6], int enc, int obs_dtype, PlaneTab out[2][3]) {
    int8_t tab[2 * 3 * 8];
    const int LP = tron_build_plane_tables(lut6, enc, tab);
    for (int p = 0; p < 2; ++p)
        for (int q = 0; q < 3; ++q) {
            uint8_t lo[8] = {0}, hi[8] = {0};
            if (q < LP)
                for (int tile = -1; tile <= 6; ++tile) {
                    const int v = tab[(p * LP + q) * 8 + (tile + 1)];
                    const int di = tile & 7;
                    if (obs_dtype == TRON_I8) { lo[di] = (uint8_t)(int8_t)v; }
                    else { const uint16_t b = bf16_bits_of_int8(v); lo[di] = (uint8_t)(b & 0xFF); hi[di] = (uint8_t)(b >> 8); }
                }
            memcpy(&out[p][q].lo0, lo, 4); memcpy(&out[p][q].lo1, lo + 4, 4);
            memcpy(&out[p][q].hi0, hi, 4); memcpy(&out[p][q].hi1, hi + 4, 4);
        }
}

int fill_params(const tron_step_args* a, int mode, StepParams& p) {
    if (!a || a->struct_size != sizeof(tron_step_args)) return TRON_ERR_INVALID;
    if (!geometry_ok(a->n_envs, a->width, a->height) || !a->state) return TRON_ERR_INVALID;
    if (!layout_known(a->layout)) return TRON_ERR_INVALID;
    if (!layout_ok(a->layout, a->width, a->height)) return TRON_ERR_UNSUPPORTED;
    if (a->slide_mode < TRON_SLIDE_NONE || a->slide_mode > TRON_SLIDE_TEMPER) return TRON_ERR_INVALID;
    if (a->layout == TRON_LAYOUT_BITS10 && mode == MODE_STEP && a->slide_mode != TRON_SLIDE_NONE) return TRON_ERR_UNSUPPORTED;
    if (((uintptr_t)a->state & 15u) != 0) return TRON_ERR_ALIGN;
    memset(&p, 0, sizeof p);
    p.N = a->n_envs; p.W = a->width; p.H = a->height; p.Hc = a->height + 2; p.C = (a->width + 2) * (a->height + 2);
    p.layout = a->layout;
    p.grid = (int8_t*)a->state;
    p.meta = (uint2*)((char*)a->state + align256((size_t)p.N * grid_stride(a->layout, a->width, a->height)));
    p.boxes = (uint2*)((char*)p.meta + align256((size_t)p.N * sizeof(tron_meta)));
    p.state_off = 0; p.state_N = p.N;
    p.variant = (int)g_encode_variant;
    p.T = 1; p.obs_every_tick = 1;
    const int planes = planes_of(a->obs_enc);
    if (a->obs_enc != TRON_ENC_NONE && mode != MODE_RESET) {
        if (!planes || !a->obs) return TRON_ERR_INVALID;
        if (a->obs_dtype != TRON_BF16 && a->obs_dtype != TRON_F32 && a->obs_dtype != TRON_I8) return TRON_ERR_INVALID;
        if (((uintptr_t)a->obs & 15u) != 0) return TRON_ERR_ALIGN;
        p.obs = a->obs; p.P = planes; p.const_plane = a->const_plane; p.obs_es = tron_elem(a->obs_dtype);
        build_device_tables(a->lut, a->obs_enc, a->obs_dtype, p.tab);
    } else if (mode == MODE_OBSERVE) {
        return TRON_ERR_INVALID;
    }
    if (a->extra) {  // [degree, weight_p] side features come from the per-game temper parameters
        if (!a->slide_params) return TRON_ERR_INVALID;
        if (((uintptr_t)a->extra & 15u) != 0) return TRON_ERR_ALIGN;
        p.extra = a->extra;
    }
    p.slide_params = a->slide_params;
    p.slide_mode = a->slide_mode;
    if (a->slide_mode == TRON_SLIDE_TEMPER && !a->slide_params && mode != MODE_OBSERVE) return TRON_ERR_INVALID;
    if (a->spawn_mode != TRON_SPAWN_UNIFORM && a->spawn_mode != TRON_SPAWN_FAIR) return TRON_ERR_INVALID;
    if (mode == MODE_STEP) {
        if (a->actions && a->action_dtype != TRON_U8 && a->action_dtype != TRON_I32 && a->action_dtype != TRON_I64) return TRON_ERR_INVALID;
        if (a->slide_mode == TRON_SLIDE_TAPE && !a->slide_tape) return TRON_ERR_INVALID;
        if (a->obs_terminal) {
            if (!p.obs) return TRON_ERR_INVALID;
            if (((uintptr_t)a->obs_terminal & 15u) != 0) return TRON_ERR_ALIGN;
            p.obs_term = a->obs_terminal;
        }
        p.obs_prev = (p.obs && a->obs_prev) ? 1 : 0;
        p.actions = a->actions; p.action_dtype = a->action_dtype;
        p.reward = a->reward; p.done = a->done; p.winner = a->winner; p.eplen = a->ep_len_out;
        p.slide_tape = a->slide_tape; p.stats = (unsigned long long*)a->stats;
        p.auto_reset = a->auto_reset;
        p.ice_thr = (long long)((double)a->slide_rate * 16777216.0);
        if (a->policy != TRON_POLICY_UNIFORM && a->policy != TRON_POLICY_FREE_EPS) return TRON_ERR_INVALID;
        p.eps_thr = a->policy == TRON_POLICY_FREE_EPS ? (long long)((double)a->policy_epsilon * 16777216.0) : -1;
        p.r_base = a->reward_table.step_base; p.r_tick = a->reward_table.step_per_tick;
        p.r_win = a->reward_table.win; p.r_lose = a->reward_table.lose; p.r_draw = a->reward_table.draw;
    }
    if (mode != MODE_OBSERVE) p.spawn = a->spawn;
    p.seed = a->seed; philox_expand(a->seed, p.rk); p.counter = a->counter; p.env_base = a->env_id_base; p.spawn_mode = a->spawn_mode;
    p.counter_dev = (const unsigned long long*)a->counter_dev;
    return TRON_OK;
}

void slice_params(const StepParams& base, int lo, int n, StepParams& p) {
    p = base;
    p.N = n; p.env_base = base.env_base + (unsigned long long)lo;
    if (layout_is_dense(base.layout)) p.state_off = base.state_off + lo;
    else p.grid = base.grid + (size_t)lo * grid_stride(base.layout, base.W, base.H);
    p.meta = base.meta + lo; p.boxes = base.boxes + lo;
    const size_t frame = (size_t)2 * base.P * base.C * base.obs_es;
    if (p.actions) p.actions = (const char*)base.actions + 2 * (size_t)lo * tron_elem(base.action_dtype);
    if (p.spawn) p.spawn = base.spawn + 4 * (size_t)lo;
    if (p.slide_tape) p.slide_tape = base.slide_tape + 2 * (size_t)lo;
    if (p.slide_params) p.slide_params = base.slide_params + 4 * (size_t)lo;
    if (p.env_mask) p.env_mask = base.env_mask + lo;
    if (p.obs) p.obs = (char*)base.obs + (size_t)lo * frame;
    if (p.obs_term) p.obs_term = (char*)base.obs_term + (size_t)lo * frame;
    if (p.extra) p.extra = base.extra + 4 * (size_t)lo;
    if (p.reward) p.reward = base.reward + 2 * (size_t)lo;
    if (p.done) p.done = base.done + lo;
    if (p.winner) p.winner = base.winner + lo;
    if (p.eplen) p.eplen = base.eplen + lo;
}

int dispatch(StepParams& p, int mode, int obs_dtype, int obs_enc, cudaStream_t s) {
    const int kind = mode == MODE_RESET ? 0 : enc_kind_of(obs_enc);
    if (p.layout == TRON_LAYOUT_BITS10) return launch_step_bits10(p, mode, obs_dtype, kind, s);
    if (p.layout == TRON_LAYOUT_BITS) return launch_step_bits(p, mode, obs_dtype, kind, s);
    if (p.layout == TRON_LAYOUT_TRAIL) return (kind == 0 || mode == MODE_RESET) ? launch_step_trail(p, mode, s) : launch_step_trail_obs(p, mode, obs_dtype, kind, s);
    if (mode == MODE_STEP && kind == 0 && p.C >= g_sparse_min_cells) return launch_step_sparse(p, s);
    if (p.C == 144 && p.Hc == 12) { p.G = tile_envs_c144(p.N); return launch_step_c144(p, mode, obs_dtype, kind, s); }
    p.G = tile_envs_generic(p.C);
    return launch_step_generic(p, mode, obs_dtype, kind, s);
}

// geometry-only parameter block for the export / import kernels of the dense layouts
static void geometry_params(void* state, int n, int w, int h, int layout, StepParams& p) {
    memset(&p, 0, sizeof p);
    p.N = n; p.W = w; p.H = h; p.Hc = h + 2; p.C = (w + 2) * (h + 2); p.layout = layout;
    p.grid = (int8_t*)state; p.state_off = 0; p.state_N = n;
    p.meta = (uint2*)((char*)state + align256((size_t)n * grid_stride(layout, w, h)));
}

}  // namespace tron

extern "C" {

int tron_abi_version(void) { return TRON_B200_ABI_VERSION; }

const char* tron_status_string(int status) {
    switch (status) {
        case TRON_OK: return "ok";
        case TRON_ERR_INVALID: return "invalid argument";
        case TRON_ERR_UNSUPPORTED: return "unsupported";
        case TRON_ERR_CUDA: return "CUDA error (no usable device or launch failure); there is no CPU fallback";
        case TRON_ERR_ALIGN: return "misaligned pointer";
        default: return "unknown status";
    }
}

int tron_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return TRON_ERR_CUDA; }
    return n;
}

int tron_cells_per_env(int width, int height) { return (width + 2) * (height + 2); }
int tron_enc_planes(int obs_enc) { return planes_of(obs_enc); }
int tron_dtype_size(int dtype) { return tron_elem(dtype); }

int tron_state_offsets(int n_envs, int width, int height, int layout, size_t* grid_off, size_t* meta_off, size_t* boxes_off) {
    if (!geometry_ok(n_envs, width, height) || !layout_known(layout)) return TRON_ERR_INVALID;
    if (!layout_ok(layout, width, height)) return TRON_ERR_UNSUPPORTED;
    const size_t mo = align256((size_t)n_envs * grid_stride(layout, width, height));
    if (grid_off) *grid_off = 0;
    if (meta_off) *meta_off = mo;
    if (boxes_off) *boxes_off = mo + align256((size_t)n_envs * sizeof(tron_meta));
    return TRON_OK;
}
int tron_state_bytes(int n_envs, int width, int height, int layout, size_t* total_bytes) {
    size_t bo = 0;
    const int rc = tron_state_offsets(n_envs, width, height, layout, nullptr, nullptr, &bo);
    if (rc != TRON_OK || !total_bytes) return rc != TRON_OK ? rc : TRON_ERR_INVALID;
    *total_bytes = bo + (size_t)n_envs * 8u;
    return TRON_OK;
}
int tron_set_option(int option, int64_t value) {
    if (option == TRON_OPT_SPARSE_MIN_CELLS && value >= 0) { g_sparse_min_cells = value; return TRON_OK; }
    if (option == TRON_OPT_TILE_BYTES && value >= 1024 && value <= 200 * 1024) { tron::g_tile_bytes = value; return TRON_OK; }
    if (option == TRON_OPT_ENCODE_VARIANT && value >= 0 && value < 256) { g_encode_variant = value; return TRON_OK; }
    if (option == TRON_OPT_BITS_CTAS_PER_SM && value >= 0 && value <= 32) { g_bits_ctas_per_sm = value; return TRON_OK; }
    if (option == TRON_OPT_TILE_CTAS_PER_SM && value >= 0 && value <= 32) { g_tile_ctas_per_sm = value; return TRON_OK; }
    return TRON_ERR_INVALID;
}

// reference tron/map.py:67-81 (colour table) and tron/util.py:11-37 (pop_up applied to the colour value)
int tron_build_plane_tables(const int8_t lut6_in[6], int obs_enc, int8_t* tab) {
    static const int8_t dflt[6] = {1, -1, -2, -3, 10, -10};
    if (!lut6_in || !tab || !planes_of(obs_enc)) return TRON_ERR_INVALID;
    int8_t lut6[6];
    bool allzero = true;
    for (int i = 0; i < 6; ++i) allzero = allzero && lut6_in[i] == 0;
    memcpy(lut6, allzero ? dflt : lut6_in, 6);
    const int LP = obs_enc == TRON_ENC_LUT1 ? 1 : 3;
    for (int p = 0; p < 2; ++p) {
        int8_t col[8];
        col[TRON_TILE_WALL + 1] = lut6[1];
        col[TRON_TILE_EMPTY + 1] = lut6[0];
        col[TRON_TILE_P1_BODY + 1] = col[TRON_TILE_P1_SLIDE + 1] = p == 0 ? lut6[2] : lut6[3];
        col[TRON_TILE_P2_BODY + 1] = col[TRON_TILE_P2_SLIDE + 1] = p == 0 ? lut6[3] : lut6[2];
        col[TRON_TILE_P1_HEAD + 1] = p == 0 ? lut6[4] : lut6[5];
        col[TRON_TILE_P2_HEAD + 1] = p == 0 ? lut6[5] : lut6[4];
        for (int t = 0; t < 8; ++t) {
            const int o = col[t];
            if (LP == 1) { tab[p * 8 + t] = (int8_t)o; continue; }
            tab[(p * 3 + 0) * 8 + t] = (int8_t)(o == -1);
            tab[(p * 3 + 1) * 8 + t] = (int8_t)(o == -2 ? 1 : o == 10 ? 10 : 0);
            tab[(p * 3 + 2) * 8 + t] = (int8_t)(o == -3 ? 1 : o == -10 ? 10 : 0);
        }
    }
    return LP;
}

int tron_reset(void* state, int n_envs, int width, int height, int layout, const int8_t* spawn, int spawn_mode, const uint8_t* env_mask,
               uint64_t seed, uint64_t counter, uint64_t env_id_base, tron_stream_t stream) {
    if (spawn_mode != TRON_SPAWN_UNIFORM && spawn_mode != TRON_SPAWN_FAIR) return TRON_ERR_INVALID;
    tron_step_args a;
    memset(&a, 0, sizeof a);
    a.struct_size = sizeof a; a.n_envs = n_envs; a.width = width; a.height = height; a.layout = layout; a.state = state;
    a.seed = seed; a.counter = counter; a.env_id_base = env_id_base; a.spawn_mode = spawn_mode;
    StepParams p;
    const int rc = fill_params(&a, MODE_RESET, p);
    if (rc != TRON_OK) return rc;
    p.spawn = spawn; p.env_mask = env_mask;
    return dispatch(p, MODE_RESET, TRON_I8, TRON_ENC_NONE, (cudaStream_t)stream);
}

int tron_reset_ex(const tron_step_args* args, const uint8_t* env_mask, tron_stream_t stream) {
    StepParams p;
    const int rc = fill_params(args, MODE_RESET, p);
    if (rc != TRON_OK) return rc;
    p.env_mask = env_mask;
    return dispatch(p, MODE_RESET, TRON_I8, TRON_ENC_NONE, (cudaStream_t)stream);
}

int tron_step(const tron_step_args* args, tron_stream_t stream) {
    StepParams p;
    const int rc = fill_params(args, MODE_STEP, p);
    if (rc != TRON_OK) return rc;
    return dispatch(p, MODE_STEP, args->obs_dtype, args->obs_enc, (cudaStream_t)stream);
}

int tron_step_many(const tron_step_args* args, tron_stream_t stream) {
    StepParams p;
    const int rc = fill_params(args, MODE_STEP, p);
    if (rc != TRON_OK) return rc;
    if (args->n_ticks < 1) return TRON_ERR_INVALID;
    if (args->obs_terminal && args->n_ticks > 1) return TRON_ERR_UNSUPPORTED;
    p.T = args->n_ticks; p.obs_every_tick = args->obs_every_tick;
    p.obs_prev = 0;  // tron_step only
    return dispatch(p, MODE_STEP, args->obs_dtype, args->obs_enc, (cudaStream_t)stream);
}

int tron_observe(const tron_step_args* args, tron_stream_t stream) {
    StepParams p;
    const int rc = fill_params(args, MODE_OBSERVE, p);
    if (rc != TRON_OK) return rc;
    return dispatch(p, MODE_OBSERVE, args->obs_dtype, args->obs_enc, (cudaStream_t)stream);
}

int tron_export_grid(const void* state, int n_envs, int width, int height, int layout, int8_t* tiles, int8_t* heads,
                     uint8_t* alive, uint8_t* done, uint8_t* winner, int32_t* ep_len, tron_stream_t stream) {
    size_t mo = 0;
    const int rc = tron_state_offsets(n_envs, width, height, layout, nullptr, &mo, nullptr);
    if (rc != TRON_OK || !state) return rc != TRON_OK ? rc : TRON_ERR_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    StepParams p;
    geometry_params((void*)state, n_envs, width, height, layout, p);
    if (layout == TRON_LAYOUT_TRAIL) return launch_trail_export(p, tiles, heads, alive, done, winner, ep_len, s);
    if (tiles && (layout == TRON_LAYOUT_BITS10 || layout == TRON_LAYOUT_BITS)) {
        if (launch_bits_export(p, (const char*)state + mo, tiles, s) != TRON_OK) return TRON_ERR_CUDA;
    } else if (tiles && cudaMemcpyAsync(tiles, state, (size_t)n_envs * tron_cells_per_env(width, height), cudaMemcpyDeviceToDevice, s) != cudaSuccess) {
        return TRON_ERR_CUDA;
    }
    return launch_export_meta((const char*)state + mo, n_envs, heads, alive, done, winner, ep_len, s);
}

int tron_import_grid(void* state, int n_envs, int width, int height, int layout, const int8_t* tiles, const int8_t* heads,
                     const uint8_t* alive, const uint8_t* done, const uint8_t* winner, const int32_t* ep_len, tron_stream_t stream) {
    size_t mo = 0;
    const int rc = tron_state_offsets(n_envs, width, height, layout, nullptr, &mo, nullptr);
    if (rc != TRON_OK || !state) return rc != TRON_OK ? rc : TRON_ERR_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    StepParams p;
    geometry_params(state, n_envs, width, height, layout, p);
    if (layout == TRON_LAYOUT_TRAIL) return launch_trail_import(p, tiles, heads, alive, done, winner, ep_len, s);
    if (tiles && (layout == TRON_LAYOUT_BITS10 || layout == TRON_LAYOUT_BITS)) {
        if (launch_bits_import(p, tiles, heads == nullptr, s) != TRON_OK) return TRON_ERR_CUDA;
    } else if (tiles && cudaMemcpyAsync(state, tiles, (size_t)n_envs * tron_cells_per_env(width, height), cudaMemcpyDeviceToDevice, s) != cudaSuccess) {
        return TRON_ERR_CUDA;
    }
    return launch_import_meta((char*)state + mo, n_envs, width, height, heads, alive, done, winner, ep_len, layout == TRON_LAYOUT_TILE8 ? tiles : nullptr, s);
}

int tron_random_actions(uint8_t* actions, int n_envs, uint64_t seed, uint64_t counter, const uint64_t* counter_dev, uint64_t env_id_base,
                        tron_stream_t stream) {
    if (!actions || n_envs <= 0) return TRON_ERR_INVALID;
    return launch_random_actions(actions, n_envs, seed, counter, counter_dev, env_id_base, (cudaStream_t)stream);
}
int tron_advance_counter(uint64_t* counter_dev, uint64_t delta, tron_stream_t stream) {
    if (!counter_dev) return TRON_ERR_INVALID;
    return launch_advance_counter(counter_dev, delta, (cudaStream_t)stream);
}

int tron_select_actions(const void* q, int q_dtype, int n_rows, float epsilon, uint8_t* actions, uint64_t seed, uint64_t counter,
                        const uint64_t* counter_dev, uint64_t row_id_base, tron_stream_t stream) {
    if (!q || !actions || n_rows <= 0) return TRON_ERR_INVALID;
    if (((uintptr_t)q & (q_dtype == TRON_F32 ? 15u : 7u)) != 0) return TRON_ERR_ALIGN;
    return launch_select_actions(q, q_dtype, n_rows, epsilon, actions, seed, counter, counter_dev, row_id_base, (cudaStream_t)stream);
}

int tron_minimax_actions(const int8_t* tiles, int n_envs, int width, int height, int player, int tie_mode, uint64_t seed, uint64_t counter,
                         const uint64_t* counter_dev, uint64_t env_id_base, uint8_t* actions, int32_t* values, int32_t* child_ties, tron_stream_t stream) {
    if (!tiles || !actions || !geometry_ok(n_envs, width, height) || (player != 1 && player != 2) || (tie_mode != 0 && tie_mode != 1)) return TRON_ERR_INVALID;
    if ((width + 2) * (height + 2) > 256) return TRON_ERR_UNSUPPORTED;
    return launch_minimax(tiles, n_envs, width, height, player, tie_mode, seed, counter, counter_dev, env_id_base, actions, values, child_ties, (cudaStream_t)stream);
}

int tron_pop_up(const void* obs, int obs_dtype, int64_t n_maps, int cells, void* planes, int out_dtype, tron_stream_t stream) {
    if (!obs || !planes || n_maps <= 0 || cells <= 0) return TRON_ERR_INVALID;
    if (obs_dtype != TRON_F32 && obs_dtype != TRON_BF16 && obs_dtype != TRON_I8 && obs_dtype != TRON_I32 && obs_dtype != TRON_I64) return TRON_ERR_INVALID;
    if (out_dtype != TRON_F32 && out_dtype != TRON_BF16 && out_dtype != TRON_I8) return TRON_ERR_INVALID;
    return launch_pop_up(obs, obs_dtype, n_maps, cells, planes, out_dtype, (cudaStream_t)stream);
}

static int ring_ok(const replay_ring* r) {
    if (!r || r->struct_size != sizeof(replay_ring) || r->capacity <= 0 || r->frame_elems <= 0) return 0;
    if (r->frame_dtype != TRON_BF16 && r->frame_dtype != TRON_F32 && r->frame_dtype != TRON_I8) return 0;
    return r->state && r->next_state && r->action && r->reward && r->done;
}

int replay_push(const replay_ring* ring, uint64_t cursor, const void* state, const void* next_state, const uint8_t* action,
                const float* reward, const uint8_t* done, int done_stride, int64_t n, tron_stream_t stream) {
    if (!ring_ok(ring) || !state || !next_state || !action || !reward || !done) return TRON_ERR_INVALID;
    if (n <= 0 || n > ring->capacity || (done_stride != 1 && done_stride != 2)) return TRON_ERR_INVALID;
    return launch_replay_push(ring, cursor, state, next_state, action, reward, done, done_stride, n, (cudaStream_t)stream);
}

int replay_gather(const replay_ring* ring, const int64_t* idx, int64_t k, void* out_state, void* out_next, int out_dtype,
                  int64_t* out_action, float* out_reward, float* out_done, tron_stream_t stream) {
    if (!ring_ok(ring) || !idx || k <= 0 || !out_state || !out_next || !out_action || !out_reward || !out_done) return TRON_ERR_INVALID;
    if (out_dtype != TRON_F32 && out_dtype != TRON_BF16) return TRON_ERR_INVALID;
    if ((((uintptr_t)out_state | (uintptr_t)out_next | (uintptr_t)ring->state | (uintptr_t)ring->next_state) & 15u) != 0) return TRON_ERR_ALIGN;
    return launch_replay_gather(ring, idx, k, out_state, out_next, out_dtype, out_action, out_reward, out_done, (cudaStream_t)stream);
}

int replay_sample_indices(int64_t size, int64_t k, uint64_t seed, uint64_t counter, int64_t* idx, tron_stream_t stream) {
    if (!idx || k <= 0 || k > size) return TRON_ERR_INVALID;
    return launch_replay_sample(size, k, seed, counter, idx, (cudaStream_t)stream);
}

int replay_sample_gather(const replay_ring* ring, int64_t size, int64_t k, uint64_t seed, uint64_t counter, void* out_state, void* out_next,
                         int out_dtype, int64_t* out_action, float* out_reward, float* out_done, int64_t* out_idx, tron_stream_t stream) {
    if (!ring_ok(ring) || k <= 0 || k > size || size > ring->capacity || !out_state || !out_next || !out_action || !out_reward || !out_done) return TRON_ERR_INVALID;
    if (out_dtype != TRON_F32 && out_dtype != TRON_BF16) return TRON_ERR_INVALID;
    if ((((uintptr_t)out_state | (uintptr_t)out_next | (uintptr_t)ring->state | (uintptr_t)ring->next_state) & 15u) != 0) return TRON_ERR_ALIGN;
    return launch_replay_sample_gather(ring, size, k, seed, counter, out_state, out_next, out_dtype, out_action, out_reward, out_done, out_idx,
                                       (cudaStream_t)stream);
}

int replay_frames_sample_gather(const replay_frames* fr, int64_t first_tick, int64_t n_ticks, int64_t k, uint64_t seed, uint64_t counter,
                                void* out_state, void* out_next, int out_dtype, int64_t* out_action, float* out_reward, float* out_done,
                                int64_t* out_idx, tron_stream_t stream) {
    if (!fr || fr->struct_size != sizeof(replay_frames) || fr->frame_elems <= 0 || fr->n_slots < 2 || fr->rows <= 0 || (fr->rows & 1)) return TRON_ERR_INVALID;
    if (fr->frame_dtype != TRON_BF16 && fr->frame_dtype != TRON_F32 && fr->frame_dtype != TRON_I8) return TRON_ERR_INVALID;
    if (!fr->frames || !fr->action || !fr->reward || !fr->done) return TRON_ERR_INVALID;
    if (first_tick < 0 || n_ticks <= 0 || n_ticks > fr->n_slots - 1 || k <= 0 || k > n_ticks * fr->rows) return TRON_ERR_INVALID;
    if (!out_state || !out_next || !out_action || !out_reward || !out_done) return TRON_ERR_INVALID;
    if (out_dtype != TRON_F32 && out_dtype != TRON_BF16) return TRON_ERR_INVALID;
    if ((((uintptr_t)out_state | (uintptr_t)out_next | (uintptr_t)fr->frames | (uintptr_t)fr->terminal) & 15u) != 0) return TRON_ERR_ALIGN;
    return launch_replay_frames_sample_gather(fr, first_tick, n_ticks, k, seed, counter, out_state, out_next, out_dtype, out_action, out_reward,
                                              out_done, out_idx, (cudaStream_t)stream);
}

int tron_debug_violations(uint64_t* count, int32_t* first_code) { return debug_violations(count, first_code); }

}  // extern "C"
