// common.cuh -- device helpers shared by the TRON kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tron_b200.h"

namespace tron {

// ---------------------------------------------------------------------------------------------
// Debug build (-DTRON_DEBUG, libtron_b200_debug.so, tests only): every computed cell index, trail-list position, ring slot
// and env ownership is range-checked; a violation is counted (first code kept) and the access is skipped, so a test can
// assert "no violations" instead of relying on compute-sanitizer.  Release builds compile the checks away.
// ---------------------------------------------------------------------------------------------
enum : int {
    DBG_CELL_INDEX = 1,   // cell index outside [0, C)
    DBG_TRAIL_COUNT = 2,  // trail-list position >= W*H
    DBG_RING_SLOT = 3,    // replay ring slot outside [0, capacity)
    DBG_ENV_OWNER = 4,    // a thread touched an env outside [0, N)
    DBG_HEAD_RANGE = 5,   // head coordinate outside [-1, W] x [-1, H]
    DBG_BIT_INDEX = 6,    // bit-plane index outside [0, 128)
    DBG_OBS_UNIT = 7      // observation delta: unit list slot, game or chunk outside the CTA's rows
};
#ifdef TRON_DEBUG
// one counter pair per translation unit (no relocatable device code needed); each unit registers a reader with the library
static __device__ unsigned long long g_dbg_count = 0ull;
static __device__ int g_dbg_first = 0;
__device__ __forceinline__ bool dbg_fail(int code) {
    if (atomicAdd(&g_dbg_count, 1ull) == 0ull) g_dbg_first = code;
    return false;
}
int dbg_register(int (*reader)(unsigned long long*, int*));  // misc_kernels.cu
static int dbg_read_unit(unsigned long long* c, int* f) {
    return (cudaMemcpyFromSymbol(c, g_dbg_count, sizeof *c) == cudaSuccess && cudaMemcpyFromSymbol(f, g_dbg_first, sizeof *f) == cudaSuccess) ? 0 : -1;
}
static const int g_dbg_registered = dbg_register(dbg_read_unit);
#define TRON_DCHECK(cond, code) ((cond) ? true : ::tron::dbg_fail(code))
#else
#define TRON_DCHECK(cond, code) (true)
#endif

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based RNG.  Counter = {tick counter (64b), stream id (48b) | tag | sub},
// key = seed.  One stream per global env id, so results do not depend on how envs are sharded.
// ---------------------------------------------------------------------------------------------
enum : uint32_t { TAG_ACTION = 1, TAG_SPAWN = 2, TAG_SLIDE = 3, TAG_EPS = 4, TAG_SAMPLE = 5, TAG_TEMPER = 6, TAG_FAIR = 7 };

// The ten round keys of a seed (k0 + r * 0x9E3779B9, k1 + r * 0xBB67AE85) are the same for every game of a launch: the launcher
// expands them once on the host into the kernel parameters (constant bank), which takes the two key additions per round off
// every thread's instruction stream (the trail tick kernel is instruction-bound and calls Philox twice per game-tick).
struct PhiloxKeys {
    uint32_t k[20];
};
__host__ __device__ inline void philox_expand(unsigned long long seed, PhiloxKeys& rk) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; ++r) {
        rk.k[2 * r] = k0; rk.k[2 * r + 1] = k1;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
__device__ __forceinline__ uint4 philox(const PhiloxKeys& rk, unsigned long long counter, unsigned long long stream, uint32_t tag, uint32_t sub) {
    uint32_t c0 = (uint32_t)counter, c1 = (uint32_t)(counter >> 32), c2 = (uint32_t)stream;
    uint32_t c3 = ((uint32_t)(stream >> 32) & 0xFFFFu) | ((tag & 0xFFu) << 16) | ((sub & 0xFFu) << 24);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ rk.k[2 * r]; c1 = l1; c2 = h0 ^ c3 ^ rk.k[2 * r + 1]; c3 = l0;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ uint4 philox(unsigned long long seed, unsigned long long counter,
                                        unsigned long long stream, uint32_t tag, uint32_t sub) {
    uint32_t c0 = (uint32_t)counter, c1 = (uint32_t)(counter >> 32), c2 = (uint32_t)stream;
    uint32_t c3 = ((uint32_t)(stream >> 32) & 0xFFFFu) | ((tag & 0xFFu) << 16) | ((sub & 0xFFu) << 24);
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

// make_game spawn rule (reference tron/util.py:46-84).  Uniform: 4 draws over the grid.  Fair (mode="fair", util.py:48-62): a
// random point, P1 uniform in the clipped 3x3 box around it, P2 uniform in the point-mirrored box.  Either way only
// (x1,y1) is re-drawn while the two heads coincide (util.py:76-78).
template <class Key>  // Key: the 64-bit seed or its expanded PhiloxKeys
__device__ __forceinline__ char4 rng_spawn(const Key& seed, unsigned long long counter, unsigned long long env, int W, int H, int fair) {
    int lo1x = 0, hi1x = W - 1, lo1y = 0, hi1y = H - 1, lo2x = 0, hi2x = W - 1, lo2y = 0, hi2y = H - 1;
    if (fair) {
        const uint4 q = philox(seed, counter, env, TAG_FAIR, 0);
        const int py = (int)__umulhi(q.x, (uint32_t)H), px = (int)__umulhi(q.y, (uint32_t)W);
        lo1x = max(0, px - 1); hi1x = min(W - 1, px + 1); lo1y = max(0, py - 1); hi1y = min(H - 1, py + 1);
        lo2x = W - 1 - hi1x; hi2x = W - 1 - lo1x; lo2y = H - 1 - hi1y; hi2y = H - 1 - lo1y;
    }
    uint4 r = philox(seed, counter, env, TAG_SPAWN, 0);
    int x1 = lo1x + (int)__umulhi(r.x, (uint32_t)(hi1x - lo1x + 1)), y1 = lo1y + (int)__umulhi(r.y, (uint32_t)(hi1y - lo1y + 1));
    const int x2 = lo2x + (int)__umulhi(r.z, (uint32_t)(hi2x - lo2x + 1)), y2 = lo2y + (int)__umulhi(r.w, (uint32_t)(hi2y - lo2y + 1));
    uint32_t attempt = 0;
    while (x1 == x2 && y1 == y2) {
        if (++attempt >= 64) { x1 = x1 == lo1x ? hi1x : lo1x; if (x1 == x2 && y1 == y2) y1 = y1 == lo1y ? hi1y : lo1y; break; }
        r = philox(seed, counter, env, TAG_SPAWN, attempt);
        x1 = lo1x + (int)__umulhi(r.x, (uint32_t)(hi1x - lo1x + 1)); y1 = lo1y + (int)__umulhi(r.y, (uint32_t)(hi1y - lo1y + 1));
    }
    return make_char4((signed char)x1, (signed char)y1, (signed char)x2, (signed char)y2);
}

// Game.__init__ draws (reference tron/game.py:83,87): weight x2 in [40,101], degree in [-30,30].
template <class Key>
__device__ __forceinline__ char4 rng_temper(const Key& seed, unsigned long long counter, unsigned long long env) {
    const uint4 r = philox(seed, counter, env, TAG_TEMPER, 0);
    return make_char4((signed char)(-30 + (int)__umulhi(r.z, 61u)), (signed char)(40 + (int)__umulhi(r.x, 62u)),
                      (signed char)(40 + (int)__umulhi(r.y, 62u)), 0);
}

// Head positions of a Tile.value grid (for imports that give tiles but no head array): the cell holding P1_HEAD / P2_HEAD, border
// included; a grid with P2's head only is the head-on state where both heads share the cell (P2's tile is written last,
// reference game.py:205-214).  packed = r1 | c1 << 8 | r2 << 16 | c2 << 24 as in tron_meta; returns false if no head is found.
__device__ __forceinline__ bool heads_from_tiles(const int8_t* t, int W, int H, uint32_t& packed) {
    int r1 = 0, c1 = 0, r2 = 0, c2 = 0;
    bool f1 = false, f2 = false;
    for (int i = 0; i < W + 2; ++i)
        for (int j = 0; j < H + 2; ++j) {
            const int v = t[i * (H + 2) + j];
            if (v == TRON_TILE_P1_HEAD) { r1 = i - 1; c1 = j - 1; f1 = true; }
            else if (v == TRON_TILE_P2_HEAD) { r2 = i - 1; c2 = j - 1; f2 = true; }
        }
    if (!f1 && !f2) return false;
    if (!f1) { r1 = r2; c1 = c2; }
    if (!f2) { r2 = r1; c2 = c1; }
    packed = (uint32_t)(uint8_t)r1 | ((uint32_t)(uint8_t)c1 << 8) | ((uint32_t)(uint8_t)r2 << 16) | ((uint32_t)(uint8_t)c2 << 24);
    return true;
}

// ---------------------------------------------------------------------------------------------
// Blackwell/Hopper async-proxy helpers: 1-D bulk copies (TMA engine, no tensor map) + mbarrier.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_WAIT;\n"
        "bra WAIT_LOOP;\n"
        "DONE_WAIT:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared, completion signalled on the mbarrier (bytes % 16 == 0, both addresses 16-byte aligned)
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global, tracked by the per-thread bulk group
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// make generic-proxy shared-memory writes visible to the async proxy (before a bulk store reads them)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// streaming (evict-first) 16/8-byte global stores for write-once observation planes
__device__ __forceinline__ void st_cs(uint4* p, uint4 v) { __stcs(p, v); }
__device__ __forceinline__ void st_cs(uint2* p, uint2 v) { __stcs(p, v); }

// ---------------------------------------------------------------------------------------------
// Observation encoding: a cell byte (Tile.value, -1..6) indexes an 8-entry table by (tile & 7), so
// WALL (-1) is entry 7.  Tables hold the bf16 bit pattern split into low/high bytes; PRMT looks up
// four cells per instruction.  f32 = bf16 << 16 (every int8 is exact in bf16), i8 uses `lo` only.
// ---------------------------------------------------------------------------------------------
struct PlaneTab {  // 16 bytes
    uint32_t lo0, lo1, hi0, hi1;
};

// selector for 4 cells packed in one 32-bit word: 4 nibbles = (cell & 7)
__device__ __forceinline__ uint32_t cell_selector(uint32_t w) {
    const uint32_t x = w & 0x07070707u;
    const uint32_t t = x | (x >> 4);
    return __byte_perm(t, 0u, 0x4420);
}
__device__ __forceinline__ uint32_t lut4(uint32_t t0, uint32_t t1, uint32_t sel) { return __byte_perm(t0, t1, sel); }

// ---------------------------------------------------------------------------------------------
// uniform sampling WITHOUT replacement as a keyed pseudo-random permutation of [0, size): idx[i] = pi(i).
// pi = 6-round balanced Feistel network on 2*hb bits (2^(2hb) >= size), round keys from Philox(seed; counter), with
// cycle-walking (re-apply until the value falls inside [0, size)), which restricts a permutation of the power-of-two domain to a
// permutation of [0, size).  Every index is independent of the others, so sampling needs no extra launch and no shared state.
// ---------------------------------------------------------------------------------------------
struct FeistelPerm {
    uint32_t key[6];
    uint32_t mask;
    int hb;
    unsigned long long size;
};
__device__ __forceinline__ FeistelPerm feistel_make(unsigned long long size, unsigned long long seed, unsigned long long counter) {
    FeistelPerm f;
    const uint4 a = philox(seed, counter, 0ull, TAG_SAMPLE, 0), b = philox(seed, counter, 0ull, TAG_SAMPLE, 1);
    f.key[0] = a.x; f.key[1] = a.y; f.key[2] = a.z; f.key[3] = a.w; f.key[4] = b.x; f.key[5] = b.y;
    int bits = 1;
    while (bits < 62 && (1ull << bits) < size) ++bits;
    f.hb = (bits + 1) >> 1;
    f.mask = f.hb >= 32 ? 0xFFFFFFFFu : ((1u << f.hb) - 1u);
    f.size = size;
    return f;
}
__device__ __forceinline__ uint32_t feistel_mix(uint32_t v) {
    v *= 0x85EBCA6Bu; v ^= v >> 13; v *= 0xC2B2AE35u; v ^= v >> 16;
    return v;
}
__device__ __forceinline__ unsigned long long feistel_apply(const FeistelPerm& f, unsigned long long i) {
    unsigned long long x = i;
    do {
        uint32_t L = (uint32_t)(x >> f.hb) & f.mask, R = (uint32_t)x & f.mask;
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            const uint32_t t = L ^ (feistel_mix(R ^ f.key[r]) & f.mask);
            L = R; R = t;
        }
        x = ((unsigned long long)L << f.hb) | R;
    } while (x >= f.size);
    return x;
}

// what one MODE_STEP tick of env_tick (tick_core.cuh) reports for a game.  A cell accessor that derives from TickOutSink receives
// it in g.tick_out (the state replay ring re-runs ticks and keeps the result in registers); the others compile without it.
struct TickOut {
    float2 reward;
    uint32_t done, winner;
};
struct TickOutSink {
    TickOut tick_out;
};
template <class Cells>
constexpr bool kTickOutSink = __is_base_of(TickOutSink, Cells);

// the transition that sample `row` of a window replay ring draws: u = pi(row) over the window's n_ticks * rows transitions, then
// (tick, r) = (first_tick + u / rows, u % rows).  The frame ring and the state ring both sample through this one mapping, which is
// what makes them hand out the same transitions for the same window, seed and counter.
__device__ __forceinline__ longlong2 window_transition(long long first_tick, long long n_ticks, long long rows, unsigned long long seed,
                                                       unsigned long long counter, long long row) {
    const unsigned long long u = feistel_apply(feistel_make((unsigned long long)n_ticks * (unsigned long long)rows, seed, counter),
                                               (unsigned long long)row);
    return make_longlong2(first_tick + (long long)(u / (unsigned long long)rows), (long long)(u % (unsigned long long)rows));
}

}  // namespace tron
