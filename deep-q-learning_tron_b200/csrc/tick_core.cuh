// tick_core.cuh -- one tick of ONE game, shared by the tile kernel (cells in shared memory) and the sparse
// kernel (cells in HBM).  This is the restatement of the reference's Game.next_frame + Game.step
// (tron/game.py:149-277) plus reward policy, statistics and the auto-reset decision.
#pragma once
#include "common.cuh"

namespace tron {

enum : int { MODE_STEP = 0, MODE_OBSERVE = 1, MODE_RESET = 2 };

// meta.flags bit 5: the per-player dirty boxes stored behind the meta array describe every non-template cell of
// the grid (maintained by the sparse kernel only; every other writer clears the bit).
#define TRON_FLAG_BOXES_VALID 0x20u

struct StepParams {
    int8_t* grid;
    uint2* meta;   // tron_meta, 8 bytes
    uint2* boxes;  // 8 bytes per env: {r1lo, r1hi, c1lo, c1hi, r2lo, r2hi, c2lo, c2hi} in position coordinates
    const void* actions;
    void* obs;
    float* reward;
    uint8_t* done;
    uint8_t* winner;
    int32_t* eplen;
    const int8_t* spawn;
    const uint8_t* slide_tape;
    int8_t* slide_params;
    const uint8_t* env_mask;  // MODE_RESET
    unsigned long long* stats;
    unsigned long long seed, counter, env_base;
    PhiloxKeys rk;  // round keys of `seed` (philox_expand, filled by whoever sets seed)
    const unsigned long long* counter_dev;
    long long ice_thr;
    long long eps_thr;  // TRON_POLICY_FREE_EPS: explore iff 24-bit mantissa <= eps_thr; < 0 -> uniform policy
    int N, W, H, Hc, C, G, layout;
    int T, obs_every_tick, auto_reset, slide_mode, action_dtype, spawn_mode;
    int P;  // planes written per player (lut planes + optional const plane)
    int obs_es;  // bytes per observation element
    float r_base, r_tick, r_win, r_lose, r_draw, const_plane;
    PlaneTab tab[2][3];
    void* obs_term;       // tron_step_args.obs_terminal: last frame of games that finished and were auto-reset in this call
    float* extra;         // tron_step_args.extra [N,2,2] {degree, weight_p}
    // dense (structure-of-arrays) state layouts (TRAIL hot arrays, BITS planes): the arrays hold state_N games and this launch's
    // env 0 is entry state_off, so a chunked launch (host-buffer front end) addresses the same arrays as a whole-batch launch
    long long state_off;
    int state_N;
    int variant;          // TRON_OPT_ENCODE_VARIANT
    int obs_prev;         // tron_step_args.obs_prev, cleared by the launcher when the kernel cannot use it
};

__device__ __forceinline__ int read_action(const void* actions, int dtype, size_t i) {
    if (dtype == TRON_U8) return ((const uint8_t*)actions)[i];
    if (dtype == TRON_I32) { const int v = ((const int32_t*)actions)[i]; return (v < 0 || v > 255) ? 255 : v; }
    const long long v = ((const long long*)actions)[i];
    return (v < 0 || v > 255) ? 255 : (int)v;
}

struct EnvState {
    int r1, c1, r2, c2;
    uint32_t flags;
    int k;  // ticks played in this episode
    int tr1, tc1, tr2, tc2;  // heads of the game that just finished (valid when env_tick returned true in MODE_STEP)
};
__device__ __forceinline__ EnvState unpack_meta(uint2 m) {
    EnvState e;
    e.r1 = (int8_t)(m.x & 0xFF); e.c1 = (int8_t)((m.x >> 8) & 0xFF); e.r2 = (int8_t)((m.x >> 16) & 0xFF); e.c2 = (int8_t)(m.x >> 24);
    e.flags = m.y & 0xFFu; e.k = (int)(m.y >> 16);
    e.tr1 = e.tc1 = e.tr2 = e.tc2 = 0;
    return e;
}
__device__ __forceinline__ uint2 pack_meta(const EnvState& e) {
    return make_uint2((uint32_t)(uint8_t)e.r1 | ((uint32_t)(uint8_t)e.c1 << 8) | ((uint32_t)(uint8_t)e.r2 << 16) | ((uint32_t)(uint8_t)e.c2 << 24),
                      e.flags | ((uint32_t)e.k << 16));
}

// per-player bounding boxes of every cell the player has written this episode (a player only ever writes along its own path)
struct BoxRegs {
    int lo_r[2], hi_r[2], lo_c[2], hi_c[2];
};
__device__ __forceinline__ BoxRegs unpack_boxes(uint2 b) {
    BoxRegs x;
    x.lo_r[0] = (int8_t)(b.x & 0xFF); x.hi_r[0] = (int8_t)((b.x >> 8) & 0xFF); x.lo_c[0] = (int8_t)((b.x >> 16) & 0xFF); x.hi_c[0] = (int8_t)(b.x >> 24);
    x.lo_r[1] = (int8_t)(b.y & 0xFF); x.hi_r[1] = (int8_t)((b.y >> 8) & 0xFF); x.lo_c[1] = (int8_t)((b.y >> 16) & 0xFF); x.hi_c[1] = (int8_t)(b.y >> 24);
    return x;
}
__device__ __forceinline__ uint2 pack_boxes(const BoxRegs& x) {
    return make_uint2((uint32_t)(uint8_t)x.lo_r[0] | ((uint32_t)(uint8_t)x.hi_r[0] << 8) | ((uint32_t)(uint8_t)x.lo_c[0] << 16) | ((uint32_t)(uint8_t)x.hi_c[0] << 24),
                      (uint32_t)(uint8_t)x.lo_r[1] | ((uint32_t)(uint8_t)x.hi_r[1] << 8) | ((uint32_t)(uint8_t)x.lo_c[1] << 16) | ((uint32_t)(uint8_t)x.hi_c[1] << 24));
}
__device__ __forceinline__ void box_add(BoxRegs& x, int i, int r, int c) {
    x.lo_r[i] = min(x.lo_r[i], r); x.hi_r[i] = max(x.hi_r[i], r); x.lo_c[i] = min(x.lo_c[i], c); x.hi_c[i] = max(x.hi_c[i], c);
}
__device__ __forceinline__ void box_set_spawn(BoxRegs& x, const EnvState& e) {
    x.lo_r[0] = x.hi_r[0] = e.r1; x.lo_c[0] = x.hi_c[0] = e.c1;
    x.lo_r[1] = x.hi_r[1] = e.r2; x.lo_c[1] = x.hi_c[1] = e.c2;
}

// Cell accessors: env_tick() is written against get(r,c)/put(r,c,tile) in POSITION coordinates (-1..W, -1..H).
struct ByteCells {  // int8 Tile.value grid, row-major (W+2) x (H+2), in shared memory or HBM
    int8_t* p;
    int Hc;
    int C;  // cells per game (range checks of the debug build)
    __device__ __forceinline__ int get(int r, int c) const {
        const int i = (r + 1) * Hc + c + 1;
        if (!TRON_DCHECK(i >= 0 && i < C, DBG_CELL_INDEX)) return TRON_TILE_WALL;
        return p[i];
    }
    __device__ __forceinline__ void put(int r, int c, int tile) {
        const int i = (r + 1) * Hc + c + 1;
        if (!TRON_DCHECK(i >= 0 && i < C, DBG_CELL_INDEX)) return;
        p[i] = (int8_t)tile;
    }
};

// ByteCells that also remembers what it wrote (at most two bodies, two slide tiles, two heads per tick), so that a kernel
// holding the grid in shared memory can write back just those bytes instead of the whole grid.
struct LoggedByteCells {
    int8_t* p;
    int Hc;
    int C;
    int n;
    unsigned short idx[6];
    int8_t val[6];
    __device__ __forceinline__ int get(int r, int c) const {
        const int i = (r + 1) * Hc + c + 1;
        if (!TRON_DCHECK(i >= 0 && i < C, DBG_CELL_INDEX)) return TRON_TILE_WALL;
        return p[i];
    }
    __device__ __forceinline__ void put(int r, int c, int tile) {
        const int i = (r + 1) * Hc + c + 1;
        if (!TRON_DCHECK(i >= 0 && i < C, DBG_CELL_INDEX)) return;
        p[i] = (int8_t)tile;
#pragma unroll
        for (int k = 0; k < 6; ++k)
            if (k == n) { idx[k] = (unsigned short)i; val[k] = (int8_t)tile; }
        n = min(n + 1, 6);
    }
};

// bit k set iff the neighbour of (hr, hc) in direction k is a free interior cell (no trail, no head) -- the epsilon-greedy proxy
// policy's four probes.  Cell accessors with a memory-backed part overload this to issue their loads together (TrailCells).
template <class Cells>
__device__ __forceinline__ int free_neighbours(const Cells& g, const StepParams& p, const EnvState& e, int hr, int hc) {
    int m = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int rr = hr + (k == 2) - (k == 0), cc = hc + (k == 1) - (k == 3);
        const bool fr = rr >= 0 && cc >= 0 && rr < p.W && cc < p.H && g.get(rr, cc) == TRON_TILE_EMPTY &&
                        !(rr == e.r1 && cc == e.c1) && !(rr == e.r2 && cc == e.c2);
        m |= fr ? (1 << k) : 0;
    }
    return m;
}

// One tick of the env whose cells start at `g`.  Updates `e` (fresh game state if it returns true = "rebuild this grid"),
// writes reward/done/winner/ep_len for (tick t, env) and adds to the striped statistics.  TRACK maintains the dirty boxes.
// pre_actions: the two actions already fetched (and range-folded by read_action) by a kernel that prefetches its inputs.
// FEAT: which optional paths are compiled in -- FEAT_SLIDE the ice/temper slide modes, FEAT_EPS the epsilon-greedy proxy policy.  A
// launcher picks the leanest instantiation the call allows (fewer instructions and registers for the plain tick).
enum : int { FEAT_SLIDE = 1, FEAT_EPS = 2, FEAT_ALL = 3 };
static_assert(TRON_STAT_EPISODES == 0 && TRON_STAT_P1_WINS == 1 && TRON_STAT_P2_WINS == 2 && TRON_STAT_DRAWS == 3 && TRON_STAT_EP_TICKS == 4 &&
              TRON_STAT_BAD_ACTION == 5 && TRON_STAT_ENV_STEPS == 6, "env_tick's lane-per-field statistics rely on this field order");
template <int MODE, bool TRACK, int FEAT = FEAT_ALL, class Cells>
__device__ __forceinline__ bool env_tick(Cells& g, const StepParams& p, EnvState& e, long long env, int t, int tid, BoxRegs& bx,
                                         const int* pre_actions = nullptr) {
    bool do_reset = false;
    (void)TRON_DCHECK(env >= 0 && env < p.N, DBG_ENV_OWNER);
    (void)TRON_DCHECK(e.r1 >= -1 && e.r1 <= p.W && e.c1 >= -1 && e.c1 <= p.H && e.r2 >= -1 && e.r2 <= p.W && e.c2 >= -1 && e.c2 <= p.H, DBG_HEAD_RANGE);
    const unsigned long long genv = p.env_base + (unsigned long long)env;
    const unsigned long long ctr = p.counter + (p.counter_dev ? *p.counter_dev : 0ull) + (unsigned long long)t;
    const size_t tn = (size_t)t * (size_t)p.N + (size_t)env;
    if (MODE == MODE_RESET) {
        do_reset = p.env_mask ? p.env_mask[env] != 0 : true;
    } else {
        int a1, a2;
        if (pre_actions) {
            a1 = pre_actions[0]; a2 = pre_actions[1];
        } else if (p.actions) {
            a1 = read_action(p.actions, p.action_dtype, 2 * tn);
            a2 = read_action(p.actions, p.action_dtype, 2 * tn + 1);
        } else {
            const uint4 r = philox(p.rk, ctr, genv, TAG_ACTION, 0);
            a1 = (int)(r.x >> 30); a2 = (int)(r.y >> 30);
            if ((FEAT & FEAT_EPS) && p.eps_thr >= 0 && !(e.flags & TRON_FLAG_DONE)) {  // epsilon-greedy proxy: a random FREE neighbour unless exploring
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const uint32_t w = i ? r.y : r.x;
                    int& act = i ? a2 : a1;
                    act = (int)(w & 3u);
                    if ((long long)(w >> 8) <= p.eps_thr) continue;
                    const int hr = i ? e.r2 : e.r1, hc = i ? e.c2 : e.c1;
                    const int free_mask = free_neighbours(g, p, e, hr, hc);
                    const int n_free = __popc((unsigned)free_mask);
                    if (n_free) {
                        int pick = (int)__umulhi(i ? r.w : r.z, (uint32_t)n_free);
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if ((free_mask >> k) & 1) { if (pick == 0) act = k; --pick; }
                    }
                }
            }
        }
        float rw0 = 0.f, rw1 = 0.f;
        uint32_t done = 0, winner = 0;
        int fin = 0;
        bool bad = false, stepped = false;
        if (e.flags & TRON_FLAG_DONE) {  // finished game without auto-reset stays frozen
            done = 1; winner = (e.flags >> TRON_FLAG_WINNER_SHIFT) & 3u;
        } else if (a1 > 3 || a2 > 3) {
            bad = true;
        } else {
            stepped = true;
            int r1 = e.r1, c1 = e.c1, r2 = e.r2, c2 = e.c2;
            // reference game.py:155-156: both old heads become bodies before any move
            g.put(r1, c1, TRON_TILE_P1_BODY);
            g.put(r2, c2, TRON_TILE_P2_BODY);
            // reference player.py:124-132
            const int dr1 = (a1 == 2) - (a1 == 0), dc1 = (a1 == 1) - (a1 == 3);
            const int dr2 = (a2 == 2) - (a2 == 0), dc2 = (a2 == 1) - (a2 == 3);
            r1 += dr1; c1 += dc1;
            if ((FEAT & FEAT_SLIDE) && p.slide_mode != TRON_SLIDE_NONE) {  // reference game.py:163-178
                uint4 sr = make_uint4(0, 0, 0, 0);
                if (p.slide_mode >= TRON_SLIDE_ICE) sr = philox(p.rk, ctr, genv, TAG_SLIDE, 0);
                char4 tp = make_char4(0, 0, 0, 0);
                if (p.slide_mode == TRON_SLIDE_TEMPER) tp = ((const char4*)p.slide_params)[env];
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    int& rr = i ? r2 : r1; int& cc = i ? c2 : c1;
                    const int dr = i ? dr2 : dr1, dc = i ? dc2 : dc1;
                    if (i) { rr += dr; cc += dc; }
                    if (rr >= 0 && cc >= 0 && rr < p.W && cc < p.H && g.get(rr, cc) == TRON_TILE_EMPTY) {
                        bool slip;
                        const long long mant = (long long)((i ? sr.y : sr.x) >> 8);
                        if (p.slide_mode == TRON_SLIDE_TAPE) slip = p.slide_tape[2 * tn + i] != 0;
                        else if (p.slide_mode == TRON_SLIDE_ICE) slip = mant <= p.ice_thr;
                        else {
                            const long long K = 6 * (30 - (long long)tp.x) - 700 + 10 * (long long)(i ? tp.z : tp.y);
                            slip = mant * 1000 <= K * 16777216;
                        }
                        if (slip) {
                            g.put(rr, cc, i ? TRON_TILE_P2_SLIDE : TRON_TILE_P1_SLIDE);
                            rr += dr; cc += dc;
                        }
                    }
                }
            } else {
                r2 += dr2; c2 += dc2;
            }
            // reference game.py:205-214: P1 fully resolved before P2, head written in every case
            bool al1 = e.flags & TRON_FLAG_ALIVE1, al2 = e.flags & TRON_FLAG_ALIVE2;
            const bool same = r1 == r2 && c1 == c2;
            const int t1 = g.get(r1, c1);
            const int t2 = same ? (int)TRON_TILE_P1_HEAD : g.get(r2, c2);  // P2 sees P1's freshly written head
            if (r1 < 0 || c1 < 0 || r1 >= p.W || c1 >= p.H || t1 != TRON_TILE_EMPTY) al1 = false;
            if (r2 < 0 || c2 < 0 || r2 >= p.W || c2 >= p.H || t2 != TRON_TILE_EMPTY) al2 = false;
            g.put(r1, c1, TRON_TILE_P1_HEAD);
            g.put(r2, c2, TRON_TILE_P2_HEAD);  // written second: wins a shared cell
            if (TRACK) { box_add(bx, 0, r1, c1); box_add(bx, 1, r2, c2); }
            // reference game.py:264-277
            const int n_alive = (int)al1 + (int)al2;
            if (n_alive <= 1) {
                done = 1;
                if (n_alive == 1 && !same) winner = al1 ? 1u : 2u;
            }
            e.flags = (al1 ? TRON_FLAG_ALIVE1 : 0u) | (al2 ? TRON_FLAG_ALIVE2 : 0u) | (done ? TRON_FLAG_DONE : 0u) |
                      (winner << TRON_FLAG_WINNER_SHIFT) | (TRACK ? (e.flags & TRON_FLAG_BOXES_VALID) : 0u);
            if (!done) {
                rw0 = rw1 = p.r_base + p.r_tick * (float)e.k;
            } else {
                if (winner == 0) rw0 = rw1 = p.r_draw;
                else { rw0 = winner == 1 ? p.r_win : p.r_lose; rw1 = winner == 2 ? p.r_win : p.r_lose; }
                fin = e.k + 1;
                do_reset = p.auto_reset != 0;
            }
            e.r1 = r1; e.c1 = c1; e.r2 = r2; e.c2 = c2;
            e.k += 1;
        }
        if (p.reward) ((float2*)p.reward)[tn] = make_float2(rw0, rw1);
        if (p.done) p.done[tn] = (uint8_t)done;
        if (p.winner) p.winner[tn] = (uint8_t)winner;
        if (p.eplen) p.eplen[tn] = fin;
        if (p.stats) {  // warp-aggregated counters, striped over TRON_STATS_SLOTS rows
            const unsigned am = __activemask();
            if (am == 0xFFFFFFFFu) {
                // full warp: every lane's five 0/1 contributions are summed in ONE packed reduction (6-bit fields, a warp sums to at
                // most 32 per field) and lane k adds field k of the stripe -- one RED instruction for the warp instead of seven
                const bool f = fin > 0;
                const unsigned contrib = (f && winner == 1 ? 1u : 0u) | (f && winner == 2 ? 1u << 6 : 0u) | (f && winner == 0 ? 1u << 12 : 0u) |
                                         (bad ? 1u << 18 : 0u) | (stepped ? 1u << 24 : 0u);
                const unsigned sum = __reduce_add_sync(0xFFFFFFFFu, contrib);
                const unsigned ticks = __reduce_add_sync(0xFFFFFFFFu, (unsigned)fin);
                const int lane = tid & 31;  // fields: 0 episodes, 1 P1 wins, 2 P2 wins, 3 draws, 4 episode ticks, 5 bad actions, 6 env steps
                const unsigned w1 = sum & 63u, w2 = (sum >> 6) & 63u, dr = (sum >> 12) & 63u;
                const unsigned v = lane == 0 ? w1 + w2 + dr : lane == 4 ? ticks : (sum >> (6 * (lane - (lane < 4 ? 1 : 2)))) & 63u;
                if (lane < 7 && v) atomicAdd(p.stats + (size_t)(blockIdx.x % TRON_STATS_SLOTS) * TRON_STATS_FIELDS + lane, (unsigned long long)v);
            } else {
            const unsigned m_fin = __ballot_sync(am, fin > 0), m_w1 = __ballot_sync(am, fin > 0 && winner == 1),
                           m_w2 = __ballot_sync(am, fin > 0 && winner == 2), m_bad = __ballot_sync(am, bad), m_step = __ballot_sync(am, stepped);
            const unsigned ticks = __reduce_add_sync(am, (unsigned)fin);
            if ((tid & 31) == (__ffs(am) - 1)) {
                unsigned long long* s = p.stats + (size_t)(blockIdx.x % TRON_STATS_SLOTS) * TRON_STATS_FIELDS;
                if (m_fin) {
                    atomicAdd(s + TRON_STAT_EPISODES, (unsigned long long)__popc(m_fin));
                    atomicAdd(s + TRON_STAT_P1_WINS, (unsigned long long)__popc(m_w1));
                    atomicAdd(s + TRON_STAT_P2_WINS, (unsigned long long)__popc(m_w2));
                    atomicAdd(s + TRON_STAT_DRAWS, (unsigned long long)(__popc(m_fin) - __popc(m_w1) - __popc(m_w2)));
                    atomicAdd(s + TRON_STAT_EP_TICKS, (unsigned long long)ticks);
                }
                if (m_bad) atomicAdd(s + TRON_STAT_BAD_ACTION, (unsigned long long)__popc(m_bad));
                atomicAdd(s + TRON_STAT_ENV_STEPS, (unsigned long long)__popc(m_step));
            }
            }
        }
    }
    char4 tp_now = make_char4(0, 0, 0, 0);
    bool tp_known = false;
    if (do_reset) {  // fresh game (reference game.py:70-91, util.py:70-78); the caller rebuilds the cells
        const char4 sp = p.spawn ? ((const char4*)p.spawn)[tn] : rng_spawn(p.rk, ctr, genv, p.W, p.H, p.spawn_mode);
        e.tr1 = e.r1; e.tc1 = e.c1; e.tr2 = e.r2; e.tc2 = e.c2;
        e.r1 = sp.x; e.c1 = sp.y; e.r2 = sp.z; e.c2 = sp.w;
        e.flags = TRON_FLAG_ALIVE1 | TRON_FLAG_ALIVE2 | (TRACK ? (e.flags & TRON_FLAG_BOXES_VALID) : 0u);
        e.k = 0;
        // Game.__init__ draws weight x2 and degree for every fresh game whatever the mode (reference game.py:83,87), tron_reset included
        if (p.slide_params) {
            tp_now = rng_temper(p.rk, ctr, genv);
            tp_known = true;
            ((char4*)p.slide_params)[env] = tp_now;
        }
    }
    if (p.extra && p.slide_params && (MODE != MODE_STEP || t == p.T - 1)) {  // [degree, weight_p] of the game the observation shows
        if (!tp_known) tp_now = ((const char4*)p.slide_params)[env];
        ((float4*)p.extra)[env] = make_float4((float)tp_now.x, (float)tp_now.y, (float)tp_now.x, (float)tp_now.z);
    }
    return do_reset;
}

// tron_observe: the side features of the current games (no tick runs in MODE_OBSERVE)
__device__ __forceinline__ void emit_extra(const StepParams& p, long long env) {
    if (p.extra && p.slide_params) {
        const char4 tp = ((const char4*)p.slide_params)[env];
        ((float4*)p.extra)[env] = make_float4((float)tp.x, (float)tp.y, (float)tp.x, (float)tp.z);
    }
}

}  // namespace tron
