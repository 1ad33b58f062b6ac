// step_trail.cu -- ticks for LARGE grids on a TRAIL-LIST state (TRON_LAYOUT_TRAIL).
//
// A dense 64x64 grid is 4,356 B per game of which a tick touches ~6 cells scattered over several DRAM rows; the int8 sparse
// kernel is therefore bound by random 32-byte DRAM operations (~15 per game-tick), not by bandwidth.  Here a game is
//     header  16 B : tron_meta (heads, alive/done/winner flags, ep_len) | n1 u16 | n2 u16 | 4 B reserved
//     list         : the trail cells both players left behind, interleaved by player: word k = {entry (k, P1), entry (k, P2)},
//                    an entry = 2 bytes {p0 | slide<<7, p1}; capacity W*H entries per player (trail cells are distinct
//                    interior cells), so the representation is exact for any episode.
// Walls are implicit and heads live in the header.  "Is this cell free?" is a scan of both lists -- a handful of entries for
// typical episodes -- and a reset is n1 = n2 = 0.
//
// Memory layout (round 2): the header and list words 0..11 of EVERY game -- 64 "hot" bytes -- are four dense uint4 arrays
// hot[q][state_N] (q = 0 header, q = 1..3 list words 4(q-1)..4(q-1)+3); list words >= 12 live in a per-game cold area behind
// them.  A tick of thread-per-game is then four fully coalesced 512-byte warp loads, one coalesced header store and one
// coalesced store of the uint4 that received this tick's entries: the kernel streams at HBM bandwidth instead of paying one
// DRAM row activation per game (round 1 kept a game's record contiguous, 16 KB apart from its neighbours: 0.34 of peak).
// Only episodes longer than 12 ticks touch the cold area, which holds two things per game: the list words >= 12 (write-only for
// the tick: they give export / observation rendering the owner and slide flag of every cell) and an OCCUPANCY BITMAP over the
// interior cells with one bit per cell that a cold entry names.  "Is this cell free?" for a long game is then the 12-word register
// scan plus ONE 4-byte probe of the bitmap instead of a walk over the whole list (round 2 first walked it: every probe of a long
// game cost O(episode length) loads, the epsilon-greedy streams ran at a ninth of the short-episode rate); a reset of a game that
// had cold entries zeroes its bitmap (512 B at 64x64, 16-byte stores).  Unused entries of the hot words hold the impossible key
// 0xFFFF (see TrailCells), which makes "is this cell free?" a branch-free packed-minimum over the words (VIMNMX3.U16x2, 1.5
// instructions per list word); the kernel is instruction-issue-bound, not bandwidth-bound (profiles/r2_step_trail_64x64_2M.json:
// issue active 74 %, DRAM 19 %), so instruction count is what the layout and these tricks buy.
#include <algorithm>

#include "step_dispatch.cuh"

namespace tron {

constexpr int kTrailThreads = 128;
constexpr int kTrailHot = 12;  // list words held in the hot arrays / in registers (entries 0..11 of both players)

// cold area of a game: list words 12.. (lw words), then the occupancy bitmap of the cells those words name (W rows of wpr words)
__host__ __device__ inline int trail_list_words(int W, int H) {
    const int n = W * H - kTrailHot;
    return n <= 0 ? 0 : ((n + 3) & ~3);
}
__host__ __device__ inline int trail_bitmap_wpr(int H) { return (H + 31) >> 5; }
__host__ __device__ inline int trail_bitmap_words(int W, int H) { return W * H <= kTrailHot ? 0 : ((W * trail_bitmap_wpr(H) + 3) & ~3); }
__host__ __device__ inline int trail_cold_words(int W, int H) { return trail_list_words(W, H) + trail_bitmap_words(W, H); }
size_t trail_game_bytes_host(int W, int H) { return 64u + 4u * (size_t)trail_cold_words(W, H); }

// address of list word k of the game at dense index i
struct TrailStore {
    uint4* hot;
    uint32_t* cold;
    long long SN;  // games in the arrays
    int cw;        // cold words per game (list words 12.. + bitmap)
    int lw;        // of which list words
    __device__ __forceinline__ uint32_t* word(long long i, int k) const {
        return k < kTrailHot ? ((uint32_t*)(hot + (long long)(1 + (k >> 2)) * SN + i) + (k & 3)) : (cold + i * cw + (k - kTrailHot));
    }
};
__host__ __device__ inline TrailStore trail_store(const StepParams& p) {
    TrailStore s;
    s.hot = (uint4*)p.grid;
    s.SN = p.state_N;
    s.cw = trail_cold_words(p.W, p.H);
    s.lw = trail_list_words(p.W, p.H);
    s.cold = (uint32_t*)((char*)p.grid + 64ull * (unsigned long long)p.state_N);
    return s;
}

// exact per-half "is zero" test of a 32-bit word holding two 16-bit entries: bit 15 / bit 31 of the result is set iff the
// low / high half of x is zero (the top bit of each half is masked before the add, so no carry crosses the halves)
__device__ __forceinline__ uint32_t zero_halves(uint32_t x) {
    const uint32_t t = (x & 0x7FFF7FFFu) + 0x7FFF7FFFu;
    return ~(t | x | 0x7FFF7FFFu);
}

struct TrailCells {
    // list words 0..11 in registers.  INVARIANT of the hot arrays (memory and registers): an entry at a position >= n holds the
    // impossible key 0xFFFF, so that get() needs no validity test per entry.  Whoever empties a list (reset, auto-reset, import)
    // writes the placeholders back; the cold words (positions >= 12) carry no such guarantee and are tested against n.
    uint32_t hot[kTrailHot];
    uint32_t* cold;           // this game's cold words: list words 12.., then the occupancy bitmap of the cells they name
    int n0, n1;               // entries per player at the start of the tick (those are in hot[] / cold[])
    uint32_t fb, fs;          // entries appended during this tick: bodies {P1 | P2 << 16} and slide tiles, 0xFFFF = none
    int W, H;
    unsigned dirty;           // bit q: hot uint4 q changed

    __device__ __forceinline__ uint32_t* bmp() const { return cold + trail_list_words(W, H); }
    __device__ __forceinline__ int wpr() const { return trail_bitmap_wpr(H); }
    // a cold entry was appended: its cell goes into the bitmap
    __device__ __forceinline__ void mark(uint32_t entry) {
        const int r = (int)(entry & 0x7Fu), c = (int)((entry >> 8) & 0xFFu);
        const int w = r * wpr() + (c >> 5);
        const bool in_range = r < W && c < H && w < trail_bitmap_words(W, H);  // checked in release builds too: this is the rare path
        if (!TRON_DCHECK(in_range, DBG_CELL_INDEX) || !in_range) return;
        // result unused -> RED.OR: no load the tick would have to wait for.  The reduction is performed in L2 and leaves a copy of the
        // line in this SM's L1 stale, so every READ of the bitmap bypasses L1 (__ldcg): a later tick of the same launch (step_many)
        // must see the bit (found by the differential fuzz: a missed collision let a list outgrow its capacity).
        atomicOr(bmp() + w, 1u << (c & 31));
    }
    // a finished game that had cold entries: zero its bitmap (16-byte stores; the cold area of a game is 16-byte aligned and both of
    // its parts are multiples of 16 bytes).  Deliberately independent of the list contents.
    __device__ __forceinline__ void clear_bitmap() {
        uint4* b = (uint4*)bmp();
        for (int q = 0; q < trail_bitmap_words(W, H) / 4; ++q) b[q] = make_uint4(0u, 0u, 0u, 0u);
    }
    __device__ __forceinline__ static unsigned short pack(int r, int c, bool slide) { return (unsigned short)((r & 0x7F) | (slide ? 0x80 : 0) | (c << 8)); }

    __device__ __forceinline__ void start(int a, int b) { n0 = a; n1 = b; fb = fs = 0xFFFFFFFFu; dirty = 0; }
    __device__ __forceinline__ void blank() {
#pragma unroll
        for (int w = 0; w < kTrailHot; ++w) hot[w] = 0xFFFFFFFFu;
    }
    __device__ __forceinline__ void clear() {  // fresh game: empty lists; the hot uint4s that held entries go back as placeholders
        const int used = min(kTrailHot, max(n0, n1));
        dirty |= (used > 0 ? 2u : 0u) | (used > 4 ? 4u : 0u) | (used > 8 ? 8u : 0u);
        if (max(n0, n1) > kTrailHot) clear_bitmap();
        n0 = n1 = 0; fb = fs = 0xFFFFFFFFu;
        blank();
    }
    // explicit reset: establishes every invariant whatever the memory held before (placeholders in all hot words, empty bitmap)
    __device__ __forceinline__ void reset_all() {
        clear_bitmap();
        n0 = n1 = 0; fb = fs = 0xFFFFFFFFu;
        blank();
        dirty = 0xEu;
    }

    // the register part of get(): nonzero iff an entry of this tick or of list words 0..11 names the interior cell (r, c)
    __device__ __forceinline__ uint32_t hot_hit(int r, int c) const {
        const uint32_t key = (uint32_t)(r & 0x7F) | ((uint32_t)c << 8), key2 = key | (key << 16);
        // per 16-bit half: (entry without its slide flag) ^ key is zero iff the entry is this cell; a running packed minimum
        // (VIMNMX3.U16x2, two list words per instruction) ends at zero iff any entry matched
        uint32_t acc = __vimin3_u16x2(0xFFFFFFFFu, (fb & 0xFF7FFF7Fu) ^ key2, (fs & 0xFF7FFF7Fu) ^ key2);
#pragma unroll
        for (int w = 0; w < kTrailHot; w += 2) acc = __vimin3_u16x2(acc, (hot[w] & 0xFF7FFF7Fu) ^ key2, (hot[w + 1] & 0xFF7FFF7Fu) ^ key2);
        return zero_halves(acc);
    }
    __device__ __forceinline__ int get(int r, int c) const {
        if (r < 0 || c < 0 || r >= W || c >= H) return TRON_TILE_WALL;
        uint32_t hit = hot_hit(r, c);
        if (max(n0, n1) > kTrailHot) {  // long episode: the cells of the list entries 12.. are in the bitmap
            const int w = r * wpr() + (c >> 5);
            const bool in_range = w < trail_bitmap_words(W, H);
            if (TRON_DCHECK(in_range, DBG_CELL_INDEX) && in_range) hit |= (__ldcg(bmp() + w) >> (c & 31)) & 1u;  // L2 read, see mark()
        }
        return hit ? TRON_TILE_P1_BODY : TRON_TILE_EMPTY;  // callers only test for EMPTY
    }
    __device__ __forceinline__ void put(int r, int c, int tile) {
        if (tile != TRON_TILE_P1_BODY && tile != TRON_TILE_P2_BODY && tile != TRON_TILE_P1_SLIDE && tile != TRON_TILE_P2_SLIDE) return;  // heads are metadata
        if (r < 0 || c < 0 || r >= W || c >= H) return;  // a head that left the board leaves no trail tile there
        const bool slide = tile == TRON_TILE_P1_SLIDE || tile == TRON_TILE_P2_SLIDE;
        const bool p2 = tile == TRON_TILE_P2_BODY || tile == TRON_TILE_P2_SLIDE;
        const uint32_t e = pack(r, c, slide);
        uint32_t& f = slide ? fs : fb;
        f = p2 ? ((f & 0x0000FFFFu) | (e << 16)) : ((f & 0xFFFF0000u) | e);
    }
    __device__ __forceinline__ void append(int owner, int k, uint32_t entry) {
        if (!TRON_DCHECK(k < W * H, DBG_TRAIL_COUNT) || k >= W * H) return;
        const uint32_t v = entry << (16 * owner), keep = owner ? 0x0000FFFFu : 0xFFFF0000u;
        if (k < kTrailHot) {
#pragma unroll
            for (int w = 0; w < kTrailHot; ++w)
                if (w == k) hot[w] = (hot[w] & keep) | v;
            dirty |= 1u << (1 + (k >> 2));
        } else {
            // one half of a list word: a 2-byte store in PTX, opaque to the compiler's type-based alias analysis (the word is read as 32 bits elsewhere)
            asm volatile("st.global.u16 [%0], %1;" ::"l"((unsigned short*)(cold + (k - kTrailHot)) + owner), "h"((unsigned short)entry) : "memory");
            mark(entry);
        }
    }
    // append this tick's entries to the lists (registers for list words < 12, memory beyond): per player the body, then the slide tile
    __device__ __forceinline__ void commit() {
        if (fs == 0xFFFFFFFFu && n0 == n1 && (fb & 0xFFFFu) != 0xFFFFu && (fb >> 16) != 0xFFFFu) {
            // the common tick: both players leave one body, their lists are equally long -> the two entries are ONE list word
            const int k = n0;
            if (TRON_DCHECK(k < W * H, DBG_TRAIL_COUNT) && k < W * H) {
                if (k < kTrailHot) {
#pragma unroll
                    for (int w = 0; w < kTrailHot; ++w)
                        if (w == k) hot[w] = fb;
                    dirty |= 1u << (1 + (k >> 2));
                } else {
                    cold[k - kTrailHot] = fb;
                    mark(fb & 0xFFFFu);
                    mark(fb >> 16);
                }
            }
            n0 = n1 = k + 1;
        } else {
            if ((fb & 0xFFFFu) != 0xFFFFu) append(0, n0++, fb & 0xFFFFu);
            if ((fs & 0xFFFFu) != 0xFFFFu) append(0, n0++, fs & 0xFFFFu);
            if ((fb >> 16) != 0xFFFFu) append(1, n1++, fb >> 16);
            if ((fs >> 16) != 0xFFFFu) append(1, n1++, fs >> 16);
        }
        fb = fs = 0xFFFFFFFFu;
    }
    // upto_words: list words that can hold valid entries or receive this call's appends; the others are placeholders by the invariant
    __device__ __forceinline__ void load_hot(const TrailStore& st, long long i, int upto_words) {
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            uint4 v = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
            if (4 * q < upto_words) v = st.hot[(long long)(1 + q) * st.SN + i];
            hot[4 * q] = v.x; hot[4 * q + 1] = v.y; hot[4 * q + 2] = v.z; hot[4 * q + 3] = v.w;
        }
    }
    __device__ __forceinline__ void store_dirty(const TrailStore& st, long long i) {
#pragma unroll
        for (int q = 0; q < 3; ++q)
            if (dirty & (1u << (1 + q))) st.hot[(long long)(1 + q) * st.SN + i] = make_uint4(hot[4 * q], hot[4 * q + 1], hot[4 * q + 2], hot[4 * q + 3]);
        dirty = 0;
    }
};

// The epsilon-greedy proxy policy probes the four neighbours of a head.  For a long game each probe needs one bitmap word from the
// cold area: the four loads are issued together, before any of them is used (env_tick() calls this through ADL; one after the
// other they were four dependent DRAM round trips per player and tick, and the kernel was bound by exactly that latency).
__device__ __forceinline__ int free_neighbours(const TrailCells& g, const StepParams& p, const EnvState& e, int hr, int hc) {
    const bool cold_on = max(g.n0, g.n1) > kTrailHot;
    const uint32_t* b = g.bmp();
    const int wpr = g.wpr();
    int rr[4], cc[4];
    bool inb[4];
    uint32_t wv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        rr[k] = hr + (k == 2) - (k == 0); cc[k] = hc + (k == 1) - (k == 3);
        inb[k] = rr[k] >= 0 && cc[k] >= 0 && rr[k] < g.W && cc[k] < g.H;
        const int w = rr[k] * wpr + (cc[k] >> 5);
        wv[k] = 0u;
        const bool in_range = w >= 0 && w < trail_bitmap_words(g.W, g.H);
        if (cold_on && inb[k] && TRON_DCHECK(in_range, DBG_CELL_INDEX) && in_range) wv[k] = __ldcg(b + w);  // L2 read, see mark()
    }
    int m = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (!inb[k]) continue;
        const uint32_t hit = g.hot_hit(rr[k], cc[k]) | ((wv[k] >> (cc[k] & 31)) & 1u);
        const bool fr = !hit && !(rr[k] == e.r1 && cc[k] == e.c1) && !(rr[k] == e.r2 && cc[k] == e.c2);
        m |= fr ? (1 << k) : 0;
    }
    return m;
}

// 64 registers (8 CTAs per SM): the kernel is issue-bound and the extra warps beat the 16 bytes of spill this costs (measured: an
// 80-register build without spills is 7 % slower)
template <int MODE, int FEAT>
__global__ void __launch_bounds__(kTrailThreads, 8) step_trail_kernel(const StepParams p) {
    const int tid = threadIdx.x;
    const long long env = (long long)blockIdx.x * kTrailThreads + tid;
    if (env >= p.N) return;
    const TrailStore st = trail_store(p);
    const long long i = p.state_off + env;
    const uint4 hdr = st.hot[i];
    EnvState e = unpack_meta(make_uint2(hdr.x, hdr.y));
    TrailCells g;
    g.W = p.W; g.H = p.H; g.cold = st.cold + i * st.cw;
    g.start((int)(hdr.z & 0xFFFFu), (int)(hdr.z >> 16));
    if (MODE == MODE_STEP) {
        // a list word beyond max(n0, n1) holds nothing valid and a tick appends at most two entries per player, so only the
        // uint4s up to word max(n) + 2T are fetched (one 16-byte load for young games; the others are placeholders by the invariant)
        g.load_hot(st, i, min(kTrailHot, max(g.n0, g.n1) + 2 * p.T));
    } else {
        g.blank();  // MODE_RESET never looks at the lists; games that are not reset keep theirs
    }
    const int T = MODE == MODE_STEP ? p.T : 1;
    for (int t = 0; t < T; ++t) {
        BoxRegs bx;
        const bool do_reset = env_tick<MODE, false, FEAT>(g, p, e, env, t, tid, bx);
        if (do_reset) {
            if (MODE == MODE_RESET) g.reset_all();
            else g.clear();
        } else {
            g.commit();
        }
    }
    const uint2 m = pack_meta(e);
    st.hot[i] = make_uint4(m.x, m.y, (uint32_t)g.n0 | ((uint32_t)g.n1 << 16), 0u);
    g.store_dirty(st, i);  // MODE_RESET: the placeholders of the games that were reset
}

// ---- fused tick + observation planes on the trail-list state ------------------------------------------------------------
// Almost every cell of a game is template (border WALL, interior EMPTY), so no per-game grid is materialised at all:
//   1. thread-per-game ticks the records (up to 128 games per CTA, every lane busy);
//   2. each warp then takes its own 32 games one after the other (state broadcast with shuffles): all 32 lanes stream the
//      TEMPLATE observation of that game -- the shared template tile in shared memory pushed through the PRMT encoder,
//      full-sector coalesced streaming stores -- then, after __syncwarp(), overwrite the handful of trail cells and the two
//      heads with scattered element stores that still hit L2.
// HBM traffic per game-tick: the observation planes + one 64-byte record head; no grid read, no write-back, no
// block-wide barrier after the template is built.
template <int OD>
__device__ __forceinline__ void store_elem(char* plane, int cell, const PlaneTab& t, int tile) {
    const int sh = 8 * (tile & 7);
    const unsigned long long lo = ((unsigned long long)t.lo1 << 32) | t.lo0, hi = ((unsigned long long)t.hi1 << 32) | t.hi0;
    const uint32_t b = (uint32_t)((lo >> sh) & 0xFFull) | ((uint32_t)((hi >> sh) & 0xFFull) << 8);
    if (OD == TRON_BF16) ((unsigned short*)plane)[cell] = (unsigned short)b;
    else if (OD == TRON_F32) ((uint32_t*)plane)[cell] = b << 16;
    else ((unsigned char*)plane)[cell] = (unsigned char)(b & 0xFFu);
}

template <int OD, int LP, bool CP, int CH, int MODE>
__global__ void __launch_bounds__(kTrailThreads) step_trail_obs_kernel(const StepParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int ES = OD == TRON_F32 ? 4 : OD == TRON_BF16 ? 2 : 1;
    const int C = p.C, G = p.G, Hc = p.Hc, tid = threadIdx.x, lane = tid & 31, P = p.P;
    int8_t* tmpl = (int8_t*)smem_raw;  // [C] template Tile.values shared by every game of the CTA
    const long long env0 = (long long)blockIdx.x * G;
    const int nG = (int)min((long long)G, (long long)p.N - env0);
    for (int c = tid; c < ((C + 3) & ~3); c += blockDim.x) {
        const int r = c / Hc, q = c - r * Hc;
        tmpl[c] = (c >= C || r == 0 || r == p.W + 1 || q == 0 || q == p.H + 1) ? (int8_t)TRON_TILE_WALL : (int8_t)TRON_TILE_EMPTY;
    }
    // each of the 4 warps owns gpw = G/4 consecutive games (lanes 0..gpw-1 tick them); few games per warp keep the serial
    // per-warp streaming loop short so that the grid has many waves (32 games per warp left a 1.7-wave tail: -15 %)
    const int gpw = G >> 2, warp = tid >> 5;
    const int local = warp * gpw + lane;
    const bool owner = lane < gpw && local < nG;
    const long long env = env0 + local;
    const TrailStore st = trail_store(p);
    const long long gi = p.state_off + (owner ? env : env0);
    EnvState e = unpack_meta(make_uint2(0, 0));
    TrailCells g;
    g.W = p.W; g.H = p.H; g.cold = st.cold + gi * st.cw;
    g.start(0, 0);
    g.blank();
    if (owner) {
        const uint4 hdr = st.hot[gi];
        e = unpack_meta(make_uint2(hdr.x, hdr.y));
        g.start((int)(hdr.z & 0xFFFFu), (int)(hdr.z >> 16));
        if (MODE == MODE_STEP) g.load_hot(st, gi, kTrailHot);
        if (MODE == MODE_OBSERVE) emit_extra(p, env);
    }
    __syncthreads();
    const int T = MODE == MODE_STEP ? p.T : 1;
    for (int t = 0; t < T; ++t) {
        if (MODE == MODE_STEP && owner) {
            BoxRegs bx;
            if (env_tick<MODE_STEP, false>(g, p, e, env, t, tid, bx)) g.clear();
            else g.commit();
        }
        if (!(MODE == MODE_OBSERVE || p.obs_every_tick || t == T - 1)) continue;
        if (MODE == MODE_STEP && owner) g.store_dirty(st, gi);  // the whole warp reads the lists back from memory below
        const size_t tick_off = (MODE == MODE_STEP && p.obs_every_tick) ? (size_t)t * (size_t)p.N * 2 * (size_t)P * (size_t)C * ES : 0;
        char* obase = (char*)p.obs + tick_off;
        __syncwarp();  // the entries appended in this tick (plain global stores of the owning lanes) are read by the whole warp below
        for (int src = 0; src < gpw; ++src) {  // warp-uniform loop over this warp's games
            if (warp * gpw + src >= nG) break;
            const long long senv = env0 + warp * gpw + src;
            const int n1 = __shfl_sync(0xFFFFFFFFu, g.n0, src), n2 = __shfl_sync(0xFFFFFFFFu, g.n1, src);
            const int hr1 = __shfl_sync(0xFFFFFFFFu, e.r1, src), hc1 = __shfl_sync(0xFFFFFFFFu, e.c1, src);
            const int hr2 = __shfl_sync(0xFFFFFFFFu, e.r2, src), hc2 = __shfl_sync(0xFFFFFFFFu, e.c2, src);
            char* gbase = obase + (size_t)senv * 2 * P * C * ES;
            // -- template planes
            if constexpr (CH >= 4) {
                const int per = C / 4;
                for (int ch = lane; ch < per; ch += 32) {
                    const uint32_t sel = cell_selector(((const uint32_t*)tmpl)[ch]);
#pragma unroll
                    for (int pl = 0; pl < 2; ++pl)
#pragma unroll
                        for (int q = 0; q < LP + (CP ? 1 : 0); ++q) {
                            uint32_t o[Enc4<OD>::WORDS];
                            if (q < LP) Enc4<OD>::run(p.tab[pl][q < LP ? q : 0], sel, o); else Enc4<OD>::fill(p.const_plane, o);
                            char* dst = gbase + ((size_t)(pl * P + q) * C + (size_t)ch * 4) * ES;
                            constexpr int NW = Enc4<OD>::WORDS;
                            if (NW == 4) st_cs((uint4*)dst, make_uint4(o[0], o[1 % NW], o[2 % NW], o[3 % NW]));
                            else if (NW == 2) st_cs((uint2*)dst, make_uint2(o[0], o[1 % NW]));
                            else *(uint32_t*)dst = o[0];
                        }
                }
            } else {
                for (int c = lane; c < C; c += 32) {
                    const int tile = tmpl[c];
                    for (int pl = 0; pl < 2; ++pl)
                        for (int q = 0; q < LP + (CP ? 1 : 0); ++q) {
                            char* plane = gbase + (size_t)(pl * P + q) * C * ES;
                            if (q < LP) store_elem<OD>(plane, c, p.tab[pl][q < LP ? q : 0], tile);
                            else { uint32_t o[Enc4<OD>::WORDS]; Enc4<OD>::fill(p.const_plane, o);
                                   if (ES == 4) ((uint32_t*)plane)[c] = o[0]; else if (ES == 2) ((unsigned short*)plane)[c] = (unsigned short)o[0]; else ((unsigned char*)plane)[c] = (unsigned char)o[0]; }
                        }
                }
            }
            __syncwarp();
            // -- trail cells of both players (distinct cells), then the heads (P2 last, it wins a shared cell)
            const long long si = p.state_off + senv;
            const int nmax = max(n1, n2);
            for (int k = lane; k < nmax; k += 32) {
                const uint32_t v = __ldcg(st.word(si, k));  // L2 read: another lane of this warp may have appended the entry in this tick
#pragma unroll
                for (int pl2 = 0; pl2 < 2; ++pl2) {
                    if (k >= (pl2 ? n2 : n1)) continue;
                    const unsigned u = pl2 ? (v >> 16) : (v & 0xFFFFu);
                    const int cell = ((int)(u & 0x7F) + 1) * Hc + (int)(u >> 8) + 1;
                    const int tile = pl2 ? ((u & 0x80) ? TRON_TILE_P2_SLIDE : TRON_TILE_P2_BODY) : ((u & 0x80) ? TRON_TILE_P1_SLIDE : TRON_TILE_P1_BODY);
                    for (int pl = 0; pl < 2; ++pl)
                        for (int q = 0; q < LP; ++q) store_elem<OD>(gbase + (size_t)(pl * P + q) * C * ES, cell, p.tab[pl][q], tile);
                }
            }
            __syncwarp();
            if (lane == 0) {
                for (int pl = 0; pl < 2; ++pl)
                    for (int q = 0; q < LP; ++q) {
                        char* plane = gbase + (size_t)(pl * P + q) * C * ES;
                        store_elem<OD>(plane, (hr1 + 1) * Hc + hc1 + 1, p.tab[pl][q], TRON_TILE_P1_HEAD);
                        store_elem<OD>(plane, (hr2 + 1) * Hc + hc2 + 1, p.tab[pl][q], TRON_TILE_P2_HEAD);
                    }
            }
        }
    }
    if (MODE == MODE_STEP && owner) {
        const uint2 m = pack_meta(e);
        st.hot[gi] = make_uint4(m.x, m.y, (uint32_t)g.n0 | ((uint32_t)g.n1 << 16), 0u);
    }
}

static inline bool mode_is_multi(const StepParams& p) { return p.obs_every_tick && p.T > 1; }

// ---- fused tick + observation planes, BULK-STORE edition (the default) -----------------------------------------------------
// A game's observation row [2,P,C] equals the encoded TEMPLATE row (border WALL, interior EMPTY) except at its trail cells and
// its two heads.  Each warp keeps `grp` copies of the encoded template row back to back in shared memory (a "group buffer").
// Per group of grp consecutive games it patches those few cells IN SHARED MEMORY, hands the whole buffer to the TMA engine
// (cp.async.bulk shared -> global: a handful of instructions per group instead of one store instruction per 16 bytes per lane,
// and the DRAM sees long contiguous bursts), waits until the engine has READ the buffer, and restores the patched cells.
// grp is a power of two such that (a) grp * row is a multiple of 16 bytes -- game e always uses sub-row e % grp, so shared and
// global addresses are congruent mod 16 and ANY run of sub-rows can leave as one bulk store of its 16-byte-aligned interior plus
// at most 15 bytes of byte stores at either end (partial groups at the end of a batch, single terminal frames) -- and (b) short
// rows are batched to ~8 KB per store.  Apart from those end fragments every observation byte is written by the bulk engine,
// exactly once: no scattered element stores to HBM, no write ordering between the two proxies to reason about.
template <int OD, int LP, bool CP, int MODE>
__global__ void __launch_bounds__(kTrailThreads, 6) step_trail_obs_bulk_kernel(const StepParams p, const int grp) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int ES = OD == TRON_F32 ? 4 : OD == TRON_BF16 ? 2 : 1;
    constexpr int NP = LP + (CP ? 1 : 0);
    const int C = p.C, G = p.G, Hc = p.Hc, tid = threadIdx.x, lane = tid & 31, P = p.P, warp = tid >> 5, nwarp = (int)blockDim.x >> 5;
    const uint32_t row = 2u * (uint32_t)P * (uint32_t)C * ES;        // bytes of one game's observations
    const uint32_t wbytes = ((uint32_t)grp * row + 15u) & ~15u;      // one warp's group buffer
    char* my = (char*)smem_raw + (size_t)warp * wbytes;
    // 1. the encoded template row: built once per CTA (sub-row 0 of warp 0), then replicated into every sub-row of every warp
    if ((C & 3) == 0) {
        for (int ch = tid; ch < C / 4; ch += (int)blockDim.x) {
            const int c0 = ch * 4;
            uint32_t cells = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = c0 + j, r = c / Hc, q = c - r * Hc;
                const bool wall = r == 0 || r == p.W + 1 || q == 0 || q == p.H + 1;
                cells |= (uint32_t)(uint8_t)(int8_t)(wall ? TRON_TILE_WALL : TRON_TILE_EMPTY) << (8 * j);
            }
            const uint32_t sel = cell_selector(cells);
#pragma unroll
            for (int pl = 0; pl < 2; ++pl)
#pragma unroll
                for (int q = 0; q < NP; ++q) {
                    uint32_t o[Enc4<OD>::WORDS];
                    if (q < LP) Enc4<OD>::run(p.tab[pl][q < LP ? q : 0], sel, o); else Enc4<OD>::fill(p.const_plane, o);
                    uint32_t* dst = (uint32_t*)((char*)smem_raw + ((size_t)(pl * P + q) * C + (size_t)c0) * ES);  // C % 4 == 0: 4-byte aligned
#pragma unroll
                    for (int w = 0; w < Enc4<OD>::WORDS; ++w) dst[w] = o[w];
                }
        }
    } else {
        for (int c = tid; c < C; c += (int)blockDim.x) {
            const int r = c / Hc, q0 = c - r * Hc;
            const int tile = (r == 0 || r == p.W + 1 || q0 == 0 || q0 == p.H + 1) ? TRON_TILE_WALL : TRON_TILE_EMPTY;
            for (int pl = 0; pl < 2; ++pl)
                for (int q = 0; q < NP; ++q) {
                    char* plane = (char*)smem_raw + (size_t)(pl * P + q) * C * ES;
                    if (q < LP) store_elem<OD>(plane, c, p.tab[pl][q < LP ? q : 0], tile);
                    else {
                        uint32_t o[Enc4<OD>::WORDS];
                        Enc4<OD>::fill(p.const_plane, o);
                        if (ES == 4) ((uint32_t*)plane)[c] = o[0]; else if (ES == 2) ((unsigned short*)plane)[c] = (unsigned short)o[0]; else ((unsigned char*)plane)[c] = (unsigned char)o[0];
                    }
                }
        }
    }
    __syncthreads();
    for (int j = 0; j < grp; ++j) {
        if (warp == 0 && j == 0) continue;
        char* dst = my + (size_t)j * row;
        if ((row & 3u) == 0) for (uint32_t o = (uint32_t)lane * 4u; o < row; o += 128u) *(uint32_t*)(dst + o) = *(const uint32_t*)((const char*)smem_raw + o);
        else for (uint32_t o = (uint32_t)lane; o < row; o += 32u) dst[o] = ((const char*)smem_raw)[o];
    }
    fence_proxy_async();  // every writer orders its generic-proxy writes before the bulk engine's reads
    __syncthreads();      // warp 0 must not patch its buffer while the others still copy from it

    const long long env0 = (long long)blockIdx.x * G;
    const int nG = (int)min((long long)G, (long long)p.N - env0);
    const int gpw = G / nwarp;  // a multiple of grp (launcher)
    const int local = warp * gpw + lane;
    const bool owner = lane < gpw && local < nG;
    const long long env = env0 + local;
    const TrailStore st = trail_store(p);
    const long long gi = p.state_off + (owner ? env : env0);
    EnvState e = unpack_meta(make_uint2(0, 0));
    TrailCells g;
    g.W = p.W; g.H = p.H; g.cold = st.cold + gi * st.cw;
    g.start(0, 0);
    g.blank();
    if (owner) {
        const uint4 hdr = st.hot[gi];
        e = unpack_meta(make_uint2(hdr.x, hdr.y));
        g.start((int)(hdr.z & 0xFFFFu), (int)(hdr.z >> 16));
        if (MODE == MODE_STEP) g.load_hot(st, gi, kTrailHot);
        if (MODE == MODE_OBSERVE) emit_extra(p, env);
    }
    // the 32 lanes are split evenly over the grp sub-rows: lane -> (sub-row j, position `sub` among the lpg lanes of that sub-row)
    const int lpg = 32 / grp, j = lane / lpg, sub = lane - j * lpg;
    char* mine = my + (size_t)j * row;
    auto patch = [&](int cell, int tile) {  // value of `tile` on every lut plane of this lane's sub-row
#pragma unroll
        for (int pl = 0; pl < 2; ++pl)
#pragma unroll
            for (int q = 0; q < LP; ++q) store_elem<OD>(mine + (size_t)(pl * P + q) * C * ES, cell, p.tab[pl][q], tile);
    };
    auto cell_of = [&](unsigned u) { return ((int)(u & 0x7F) + 1) * Hc + (int)(u >> 8) + 1; };
    // bytes [lo, hi) of this warp's buffer -> the same offsets behind gdst (gdst and the buffer are both 16-byte aligned)
    auto store_range = [&](uint32_t lo, uint32_t hi, char* gdst) {
        const uint32_t alo = (lo + 15u) & ~15u, ahi = hi & ~15u;
        if (alo < ahi) {
            const uint32_t chunk = (ahi - alo) >= 16384u ? 8192u : 2048u;  // bytes per lane and bulk store (profiles/r2_trail_obs_tune.jsonl)
            for (uint32_t o = alo + (uint32_t)lane * chunk; o < ahi; o += 32u * chunk) bulk_s2g(gdst + o, my + o, min(chunk, ahi - o));
            if ((uint32_t)lane < alo - lo) gdst[lo + lane] = my[lo + lane];
            if ((uint32_t)lane < hi - ahi) gdst[ahi + lane] = my[ahi + lane];
        } else {
            for (uint32_t o = lo + (uint32_t)lane; o < hi; o += 32u) gdst[o] = my[o];
        }
    };
    // One group: the games owned by lanes s0 .. s0+grp-1 of this warp; bit jj of `act` = render sub-row jj.  The per-lane arguments
    // describe the game of THIS lane's sub-row: list lengths in memory (n1 / n2), the entries of the current tick that exist only in
    // registers (fb bodies, fs slide tiles; 0xFFFF = none), the heads.  Patch, bulk-store the flagged sub-rows, wait, restore.
    auto render_group = [&](unsigned act, int s0, int n1, int n2, uint32_t fb, uint32_t fs, int hr1, int hc1, int hr2, int hc2, char* gdst) {
        const bool on = (act >> j) & 1u;
        const long long si = p.state_off + env0 + warp * gpw + s0 + j;
        const int nmax = on ? max(n1, n2) : 0;
        // L2 reads: another lane of this warp may have appended the entry in this tick; the first word per lane is kept for the restore pass
        const uint32_t v_first = sub < nmax ? __ldcg(st.word(si, sub)) : 0u;
        auto lists = [&](bool restore) {
            for (int k = sub; k < nmax; k += lpg) {
                const uint32_t v = k == sub ? v_first : __ldcg(st.word(si, k));
#pragma unroll
                for (int pl2 = 0; pl2 < 2; ++pl2) {
                    if (k >= (pl2 ? n2 : n1)) continue;
                    const unsigned u = pl2 ? (v >> 16) : (v & 0xFFFFu);
                    const int cell = cell_of(u);
                    if (!TRON_DCHECK(cell >= 0 && cell < C, DBG_CELL_INDEX)) continue;
                    patch(cell, restore ? (int)TRON_TILE_EMPTY
                                        : pl2 ? ((u & 0x80) ? TRON_TILE_P2_SLIDE : TRON_TILE_P2_BODY) : ((u & 0x80) ? TRON_TILE_P1_SLIDE : TRON_TILE_P1_BODY));
                }
            }
            if (on)
                for (int q = sub; q < 4; q += lpg) {  // the tick's own entries (terminal frames: the finished game's last bodies / slide tiles were never committed)
                    const uint32_t w = (q & 1) ? fs : fb;
                    const unsigned u = (q & 2) ? (w >> 16) : (w & 0xFFFFu);
                    if (u == 0xFFFFu) continue;
                    const int cell = cell_of(u & 0xFF7Fu);
                    if (!TRON_DCHECK(cell >= 0 && cell < C, DBG_CELL_INDEX)) continue;
                    patch(cell, restore ? (int)TRON_TILE_EMPTY
                                        : (q & 2) ? ((q & 1) ? TRON_TILE_P2_SLIDE : TRON_TILE_P2_BODY) : ((q & 1) ? TRON_TILE_P1_SLIDE : TRON_TILE_P1_BODY));
                }
        };
        // -- patch: trail cells of both players (distinct cells), then the heads (P2 last, it wins a shared cell)
        lists(false);
        __syncwarp();
        const int hcell1 = (hr1 + 1) * Hc + hc1 + 1, hcell2 = (hr2 + 1) * Hc + hc2 + 1;
        if (on && sub == 0) { patch(hcell1, TRON_TILE_P1_HEAD); patch(hcell2, TRON_TILE_P2_HEAD); }
        fence_proxy_async();  // every lane: its generic-proxy writes to the buffer become visible to the bulk engine
        __syncwarp();
        // -- every maximal run of flagged sub-rows leaves as one range
        for (unsigned m = act; m;) {
            const int a = __ffs(m) - 1;
            int b = a;
            while ((m >> b) & 1u) ++b;
            store_range((uint32_t)a * row, (uint32_t)b * row, gdst);
            m &= ~((1u << b) - 1u);
        }
        bulk_commit();
        bulk_wait_read_all();
        __syncwarp();
        // -- restore the template at the patched cells (trail cells are interior cells; a crashed head may sit on the border)
        lists(true);
        if (on && sub == 0) {
            patch(hcell1, (hr1 < 0 || hc1 < 0 || hr1 >= p.W || hc1 >= p.H) ? TRON_TILE_WALL : TRON_TILE_EMPTY);
            patch(hcell2, (hr2 < 0 || hc2 < 0 || hr2 >= p.W || hc2 >= p.H) ? TRON_TILE_WALL : TRON_TILE_EMPTY);
        }
        __syncwarp();
    };
    const unsigned FULL = 0xFFFFFFFFu;
    const int T = MODE == MODE_STEP ? p.T : 1;
    for (int t = 0; t < T; ++t) {
        bool fin = false;
        int on0 = 0, on1 = 0;
        uint32_t ofb = 0xFFFFFFFFu, ofs = 0xFFFFFFFFu;
        if (MODE == MODE_STEP && owner) {
            BoxRegs bx;
            on0 = g.n0; on1 = g.n1;
            if (env_tick<MODE_STEP, false>(g, p, e, env, t, tid, bx)) { fin = true; ofb = g.fb; ofs = g.fs; g.clear(); }
            else g.commit();
        }
        if (MODE == MODE_STEP && p.obs_term) {
            // terminal frames (tron_step_args.obs_terminal; single-tick calls only): the last frame of the games that finished in this
            // tick and were auto-reset -- their lists as they still stand in memory, this tick's uncommitted entries, the final heads
            const unsigned mfin = __ballot_sync(FULL, fin);
            for (int s0 = 0; s0 < gpw; s0 += grp) {
                const unsigned act = (mfin >> s0) & ((1u << grp) - 1u);
                if (!act) continue;
                const int sl = s0 + j;
                render_group(act, s0, __shfl_sync(FULL, on0, sl), __shfl_sync(FULL, on1, sl), __shfl_sync(FULL, ofb, sl), __shfl_sync(FULL, ofs, sl),
                             __shfl_sync(FULL, e.tr1, sl), __shfl_sync(FULL, e.tc1, sl), __shfl_sync(FULL, e.tr2, sl), __shfl_sync(FULL, e.tc2, sl),
                             (char*)p.obs_term + (size_t)(env0 + warp * gpw + s0) * row);
            }
        }
        if (!(MODE == MODE_OBSERVE || p.obs_every_tick || t == T - 1)) continue;
        if (MODE == MODE_STEP && owner) g.store_dirty(st, gi);  // the whole warp reads the lists back from memory below
        const size_t tick_off = (MODE == MODE_STEP && p.obs_every_tick) ? (size_t)t * (size_t)p.N * row : 0;
        char* obase = (char*)p.obs + tick_off;
        __syncwarp();  // the entries appended in this tick (plain global stores of the owning lanes) are read by the whole warp below
        for (int s0 = 0; s0 < gpw; s0 += grp) {  // warp-uniform loop over this warp's groups
            const int first = warp * gpw + s0;
            if (first >= nG) break;
            const int ng = min(grp, nG - first);
            const int sl = s0 + j;
            render_group((1u << ng) - 1u, s0, __shfl_sync(FULL, g.n0, sl), __shfl_sync(FULL, g.n1, sl), 0xFFFFFFFFu, 0xFFFFFFFFu,
                         __shfl_sync(FULL, e.r1, sl), __shfl_sync(FULL, e.c1, sl), __shfl_sync(FULL, e.r2, sl), __shfl_sync(FULL, e.c2, sl),
                         obase + (size_t)(env0 + first) * row);
        }
    }
    if (MODE == MODE_STEP && owner) {
        const uint2 m = pack_meta(e);
        st.hot[gi] = make_uint4(m.x, m.y, (uint32_t)g.n0 | ((uint32_t)g.n1 << 16), 0u);
    }
}

constexpr size_t kTrailBulkSmem = 200 * 1024;  // shared memory a CTA of the bulk-store kernel may use for its group buffers

template <int OD, int LP, bool CP, int MODE>
static int launch_trail_obs_one(StepParams p, cudaStream_t s) {
    const size_t es = OD == TRON_F32 ? 4 : OD == TRON_BF16 ? 2 : 1;
    const size_t row = 2 * (size_t)p.P * (size_t)p.C * es;
    // games per group: the smallest power of two that makes a group a multiple of 16 bytes, doubled while a group stays below ~8 KB
    int grp = 1;
    while ((grp * row) % 16 != 0) grp *= 2;  // <= 16: row is even
    while (grp < 16 && (size_t)grp * row < 8192) grp *= 2;
    const size_t wbytes = ((size_t)grp * row + 15) & ~(size_t)15;
    const bool ticks_aligned = !(mode_is_multi(p)) || ((size_t)p.N * row) % 16 == 0;  // every tick's block of p.obs must start 16-byte aligned
    if (!(p.variant & 32) && ((uintptr_t)p.obs & 15u) == 0 && ((uintptr_t)p.obs_term & 15u) == 0 && wbytes <= kTrailBulkSmem && ticks_aligned) {
        // as many warps (<= 4) and CTAs per SM as the shared memory holds
        const int nwarp = (int)std::min<size_t>(4, kTrailBulkSmem / wbytes);
        const size_t smem = (size_t)nwarp * wbytes;
        const int ctas_per_sm = (int)std::max<size_t>(1, std::min<size_t>(6, (size_t)(227 * 1024) / (smem + 1024)));
        // games per warp: a few waves of CTAs (the template is built once per CTA, so few, long-lived CTAs; more waves for long rows,
        // where the tail of the last wave is what costs), whole groups, at most one game per lane
        int gpw = (int)((long long)p.N / ((row >= 8192 ? 8LL : 3LL) * ctas_per_sm * sm_count() * nwarp));
        gpw = gpw > 32 ? 32 : gpw;
        gpw = gpw / grp * grp;
        gpw = gpw < grp ? grp : gpw;
        p.G = nwarp * gpw;
        const unsigned grid = (unsigned)(((long long)p.N + p.G - 1) / p.G);
        auto kernel = step_trail_obs_bulk_kernel<OD, LP, CP, MODE>;
        if (ensure_dynamic_smem((const void*)kernel, smem) != TRON_OK) return TRON_ERR_CUDA;
        kernel<<<grid, 32 * nwarp, smem, s>>>(p, grp);
        return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
    }
    if (p.obs_term) return TRON_ERR_UNSUPPORTED;  // terminal frames are rendered by the bulk-store kernel only
    // games per warp: aim at >= ~6 waves of CTAs (4 CTAs/SM resident), at most one game per lane
    int gpw = p.N / (6 * 4 * sm_count() * 4);
    gpw = gpw < 1 ? 1 : (gpw > 32 ? 32 : gpw);
    const int G = 4 * gpw;
    p.G = G;
    const size_t smem = (size_t)((p.C + 15) & ~15);
    const unsigned grid = (unsigned)(((long long)p.N + G - 1) / G);
    if ((p.C & 3) == 0) step_trail_obs_kernel<OD, LP, CP, 4, MODE><<<grid, kTrailThreads, smem, s>>>(p);
    else step_trail_obs_kernel<OD, LP, CP, 1, MODE><<<grid, kTrailThreads, smem, s>>>(p);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}
// a reset, or a step without observations (MODE_STEP / MODE_RESET only)
static int launch_trail_tick(const StepParams& p, int mode, cudaStream_t s) {
    const unsigned grid = (unsigned)(((long long)p.N + kTrailThreads - 1) / kTrailThreads);
    const bool lean = p.slide_mode == TRON_SLIDE_NONE && (p.actions != nullptr || p.eps_thr < 0);
    if (mode == MODE_STEP && lean) step_trail_kernel<MODE_STEP, 0><<<grid, kTrailThreads, 0, s>>>(p);
    else if (mode == MODE_STEP) step_trail_kernel<MODE_STEP, FEAT_ALL><<<grid, kTrailThreads, 0, s>>>(p);
    else step_trail_kernel<MODE_RESET, 0><<<grid, kTrailThreads, 0, s>>>(p);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

int launch_step_trail(const StepParams& p, int mode, int od, int enc_kind, cudaStream_t s) {
    return dispatch_obs(mode, od, enc_kind, [&](auto mode_c, auto od_c, auto lp, auto cp) {
        if constexpr (lp == 0) return launch_trail_tick(p, mode_c, s);
        else return launch_trail_obs_one<od_c, lp, cp, mode_c>(p, s);
    });
}

// ---- export: render Tile.value grids / metadata from the lists; import: rebuild the lists from grids ---------------
__global__ void trail_export_kernel(const StepParams p, int8_t* tiles, int8_t* heads, uint8_t* alive, uint8_t* done, uint8_t* winner, int32_t* ep_len) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.N) return;
    const TrailStore st = trail_store(p);
    const long long i = p.state_off + env;
    const int W = p.W, H = p.H;
    const uint4 hdr = st.hot[i];
    const EnvState e = unpack_meta(make_uint2(hdr.x, hdr.y));
    const int n1 = (int)(hdr.z & 0xFFFFu), n2 = (int)(hdr.z >> 16), Hc = H + 2, C = (W + 2) * (H + 2);
    if (tiles) {
        int8_t* t = tiles + (size_t)env * C;
        for (int c = 0; c < C; ++c) {
            const int r = c / Hc, q = c - r * Hc;
            t[c] = (r == 0 || r == W + 1 || q == 0 || q == H + 1) ? (int8_t)TRON_TILE_WALL : (int8_t)TRON_TILE_EMPTY;
        }
        for (int k = 0; k < max(n1, n2); ++k) {
            const uint32_t word = *st.word(i, k);
            for (int pl = 0; pl < 2; ++pl) {
                if (k >= (pl ? n2 : n1)) continue;
                const unsigned v = pl ? (word >> 16) : (word & 0xFFFFu);
                const int r = v & 0x7F, c = v >> 8;
                const bool slide = v & 0x80;
                t[(r + 1) * Hc + c + 1] = (int8_t)(pl ? (slide ? TRON_TILE_P2_SLIDE : TRON_TILE_P2_BODY) : (slide ? TRON_TILE_P1_SLIDE : TRON_TILE_P1_BODY));
            }
        }
        t[(e.r1 + 1) * Hc + e.c1 + 1] = TRON_TILE_P1_HEAD;
        t[(e.r2 + 1) * Hc + e.c2 + 1] = TRON_TILE_P2_HEAD;  // written second (reference game.py:205-214)
    }
    if (heads) ((uint32_t*)heads)[env] = hdr.x;
    if (alive) { alive[2 * env] = e.flags & 1u; alive[2 * env + 1] = (e.flags >> 1) & 1u; }
    if (done) done[env] = (e.flags >> 2) & 1u;
    if (winner) winner[env] = (e.flags >> TRON_FLAG_WINNER_SHIFT) & 3u;
    if (ep_len) ep_len[env] = e.k;
}
__global__ void trail_import_kernel(const StepParams p, const int8_t* __restrict__ tiles, const int8_t* heads, const uint8_t* alive, const uint8_t* done,
                                    const uint8_t* winner, const int32_t* ep_len) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.N) return;
    const TrailStore st = trail_store(p);
    const long long i = p.state_off + env;
    const int W = p.W, H = p.H;
    uint4 hdr = st.hot[i];
    if (tiles) {
        const int Hc = H + 2;
        for (int q = 1; q <= 3; ++q) st.hot[(long long)q * st.SN + i] = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);  // invariant: unused = 0xFFFF
        const int8_t* t = tiles + (size_t)env * (W + 2) * (H + 2);
        uint32_t* bmp = st.cold + i * st.cw + st.lw;
        const int wpr = trail_bitmap_wpr(H);
        for (int w = 0; w < trail_bitmap_words(W, H); ++w) bmp[w] = 0u;
        int n1 = 0, n2 = 0;
        for (int r = 0; r < W; ++r)
            for (int c = 0; c < H; ++c) {
                const int v = t[(r + 1) * Hc + c + 1];
                int k = -1;
                if (v == TRON_TILE_P1_BODY || v == TRON_TILE_P1_SLIDE) ((unsigned short*)st.word(i, k = n1++))[0] = TrailCells::pack(r, c, v == TRON_TILE_P1_SLIDE);
                else if (v == TRON_TILE_P2_BODY || v == TRON_TILE_P2_SLIDE) ((unsigned short*)st.word(i, k = n2++))[1] = TrailCells::pack(r, c, v == TRON_TILE_P2_SLIDE);
                if (k >= kTrailHot) bmp[r * wpr + (c >> 5)] |= 1u << (c & 31);  // a cold entry: its cell is looked up through the bitmap
            }
        hdr.z = (uint32_t)n1 | ((uint32_t)n2 << 16);
        uint32_t packed;
        if (!heads && heads_from_tiles(t, W, H, packed)) hdr.x = packed;  // the lists cannot hold heads: they go into the header
    }
    uint32_t f = hdr.y & 0xFFu, k = hdr.y >> 16;
    if (heads) {  // clamp to the representable range [-1, W] x [-1, H]
        const int8_t* h = heads + 4 * env;
        const int r1 = min(max((int)h[0], -1), W), c1 = min(max((int)h[1], -1), H), r2 = min(max((int)h[2], -1), W), c2 = min(max((int)h[3], -1), H);
        hdr.x = (uint32_t)(uint8_t)r1 | ((uint32_t)(uint8_t)c1 << 8) | ((uint32_t)(uint8_t)r2 << 16) | ((uint32_t)(uint8_t)c2 << 24);
    }
    if (alive) f = (f & ~3u) | (alive[2 * env] ? 1u : 0u) | (alive[2 * env + 1] ? 2u : 0u);
    if (done) f = (f & ~TRON_FLAG_DONE) | (done[env] ? TRON_FLAG_DONE : 0u);
    if (winner) f = (f & ~(3u << TRON_FLAG_WINNER_SHIFT)) | ((winner[env] & 3u) << TRON_FLAG_WINNER_SHIFT);
    if (ep_len) k = (uint32_t)ep_len[env] & 0xFFFFu;
    hdr.y = f | (k << 16);
    st.hot[i] = hdr;
}
int launch_trail_export(const StepParams& p, int8_t* tiles, int8_t* heads, uint8_t* alive, uint8_t* done, uint8_t* winner, int32_t* ep_len, cudaStream_t s) {
    trail_export_kernel<<<(p.N + 127) / 128, 128, 0, s>>>(p, tiles, heads, alive, done, winner, ep_len);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}
int launch_trail_import(const StepParams& p, const int8_t* tiles, const int8_t* heads, const uint8_t* alive, const uint8_t* done, const uint8_t* winner,
                        const int32_t* ep_len, cudaStream_t s) {
    trail_import_kernel<<<(p.N + 127) / 128, 128, 0, s>>>(p, tiles, heads, alive, done, winner, ep_len);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

}  // namespace tron
