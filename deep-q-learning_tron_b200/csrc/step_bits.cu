// step_bits.cu -- fused tick + observation on BIT-PLANE states (small boards: the reference's config.py grid and friends).
//
// Two layouts share this file:
//   TRON_LAYOUT_BITS10  10x10, no slide modes.  Per game two 128-bit planes over the 100 interior cells (bit = p0*10 + p1),
//                       `occ` (a trail tile lies here) and `own` (it belongs to player 2), stored game-major: 32 B per game.
//   TRON_LAYOUT_BITS    any W*H <= 128, every mode.  A third plane `sld` marks slide tiles (Tile 5/6, ice/temper modes,
//                       tron/game.py:163-178); the planes are three dense uint4 arrays [3][N] (48 B per game) so that every
//                       warp-wide load/store is one contiguous 512-byte run.
// Walls are implicit (the border ring), heads live in the 8-byte metadata and are overlaid when observations are encoded, a reset
// is "write zeros".  A thread keeps its game's planes in 64-bit registers: the tick is bit tests/sets, no shared-memory round
// trip.  For the observation the owning thread expands its planes into an int8 Tile.value tile in shared memory (10x10: one
// funnel-shift + bit-spread multiply per 4 cells) and the CTA runs the PRMT encode with 16-byte streaming stores.
// HBM traffic per game-tick: state read + written (32 or 48 B each way) + observation planes + ~28 B metadata.  When the caller
// says `obs` still holds the previous tick's observation (tron_step_args.obs_prev; BatchedTron.step with the buffer it wrote last),
// the 10x10 kernels with bf16 / f32 planes store only the 32-byte units whose cells this tick changed: the thread knows them from
// its pre- and post-tick planes and heads, the CTA scans the per-game counts and encodes just those units (DESIGN §4.1).
// Measured on B200 (profiles/r2_sweep.jsonl): the LINEAR store schedule below takes the 10x10 kernels from 0.94-0.97 to 0.98 of
// the measured HBM peak (pop_up 3 planes 0.95 -> 0.98, + const plane 0.94 -> 0.99); a persistent-CTA variant with register
// prefetch of the next tile was tried and dropped (0.80: it serialises the tick and store phases that otherwise overlap
// across the CTAs resident on an SM).
#include "launch.h"
#include "step_kernels.cuh"

namespace tron {

extern long long g_bits_ctas_per_sm;  // TRON_OPT_BITS_CTAS_PER_SM (abi.cu)
constexpr int kBitsThreads = 128;  // up to one game per thread; p.G games per CTA

// ------------------------------------------------------------------------------------------------ cells
template <bool SLIDE, int W_T>
struct BitCells {
    unsigned long long occ_lo, occ_hi, own_lo, own_hi, sld_lo, sld_hi;
    int Wr, Hr;  // run-time geometry, used when W_T == 0
    __device__ __forceinline__ int w() const { return W_T ? W_T : Wr; }
    __device__ __forceinline__ int h() const { return W_T ? W_T : Hr; }
    __device__ __forceinline__ int get(int r, int c) const {
        if (r < 0 || c < 0 || r >= w() || c >= h()) return TRON_TILE_WALL;
        const int b = r * h() + c;
        if (!TRON_DCHECK(b >= 0 && b < 128, DBG_BIT_INDEX)) return TRON_TILE_WALL;
        const unsigned long long o = b < 64 ? occ_lo : occ_hi, v = b < 64 ? own_lo : own_hi;
        const int occ = (int)((o >> (b & 63)) & 1ull), own = (int)((v >> (b & 63)) & 1ull);
        return occ ? (own ? TRON_TILE_P2_BODY : TRON_TILE_P1_BODY) : TRON_TILE_EMPTY;  // callers only test for EMPTY
    }
    // only trail tiles are stored: heads are metadata (overlaid at encode time), border cells are implicit
    __device__ __forceinline__ void put(int r, int c, int tile) {
        const bool body = tile == TRON_TILE_P1_BODY || tile == TRON_TILE_P2_BODY;
        const bool slide = SLIDE && (tile == TRON_TILE_P1_SLIDE || tile == TRON_TILE_P2_SLIDE);
        if (!body && !slide) return;
        if (r < 0 || c < 0 || r >= w() || c >= h()) return;
        const int b = r * h() + c;
        if (!TRON_DCHECK(b >= 0 && b < 128, DBG_BIT_INDEX)) return;
        const unsigned long long m = 1ull << (b & 63);
        const bool p2 = tile == TRON_TILE_P2_BODY || tile == TRON_TILE_P2_SLIDE;
        if (b < 64) {
            occ_lo |= m; own_lo = p2 ? (own_lo | m) : (own_lo & ~m);
            if (SLIDE) sld_lo = slide ? (sld_lo | m) : (sld_lo & ~m);
        } else {
            occ_hi |= m; own_hi = p2 ? (own_hi | m) : (own_hi & ~m);
            if (SLIDE) sld_hi = slide ? (sld_hi | m) : (sld_hi & ~m);
        }
    }
    __device__ __forceinline__ void clear() { occ_lo = occ_hi = own_lo = own_hi = sld_lo = sld_hi = 0ull; }
};

// storage: BITS10 = game-major {occ, own}; BITS = plane-major dense arrays of state_N games
template <bool SLIDE>
struct PlaneRegs {
    ulonglong2 a, b, c;
};
template <bool SLIDE>
__device__ __forceinline__ PlaneRegs<SLIDE> load_planes(const StepParams& p, long long env) {
    PlaneRegs<SLIDE> r;
    const ulonglong2* base = (const ulonglong2*)p.grid;
    if (!SLIDE) {
        r.a = base[2 * env]; r.b = base[2 * env + 1]; r.c = make_ulonglong2(0ull, 0ull);
    } else {
        const long long i = p.state_off + env;
        r.a = base[i]; r.b = base[(long long)p.state_N + i]; r.c = base[2ll * p.state_N + i];
    }
    return r;
}
template <bool SLIDE, int W_T>
__device__ __forceinline__ void store_planes(const StepParams& p, long long env, const BitCells<SLIDE, W_T>& g) {
    ulonglong2* base = (ulonglong2*)p.grid;
    if (!SLIDE) {
        base[2 * env] = make_ulonglong2(g.occ_lo, g.occ_hi);
        base[2 * env + 1] = make_ulonglong2(g.own_lo, g.own_hi);
    } else {
        const long long i = p.state_off + env;
        base[i] = make_ulonglong2(g.occ_lo, g.occ_hi);
        base[(long long)p.state_N + i] = make_ulonglong2(g.own_lo, g.own_hi);
        base[2ll * p.state_N + i] = make_ulonglong2(g.sld_lo, g.sld_hi);
    }
}
template <bool SLIDE, int W_T>
__device__ __forceinline__ void set_planes(BitCells<SLIDE, W_T>& g, const PlaneRegs<SLIDE>& r) {
    g.occ_lo = r.a.x; g.occ_hi = r.a.y; g.own_lo = r.b.x; g.own_hi = r.b.y; g.sld_lo = r.c.x; g.sld_hi = r.c.y;
}

// ------------------------------------------------------------------------------------------------ planes -> Tile.value tile
// 4 bits -> 4 bytes (bit j -> byte j): the shifted copies at 0/7/14/21 never overlap, so no carries
__device__ __forceinline__ uint32_t spread4(uint32_t n) { return ((n & 0xFu) * 0x00204081u) & 0x01010101u; }
// Tile.value bytes of 4 cells from their occ / own / slide bits: P1 body 1, P2 body 3, P1 slide 5, P2 slide 6
template <bool CODES>
__device__ __forceinline__ uint32_t tiles4(uint32_t occ4, uint32_t own4, uint32_t sld4) {
    const uint32_t o = spread4(occ4), ow = o & spread4(own4);
    uint32_t t = o + (ow << 1);
    if (CODES) {  // slide bits are a subset of occ bits: +4 for player 1, +3 for player 2 (no borrow: 4 > 1)
        const uint32_t s = spread4(sld4);
        t += (s << 2) - (s & ow);
    }
    return t;
}
__device__ __forceinline__ uint32_t row_bits10(unsigned long long lo, unsigned long long hi, int r) {  // 10 bits of interior row r
    const int b = r * 10;
    if (b + 10 <= 64) return (uint32_t)(lo >> b) & 0x3FFu;
    if (b >= 64) return (uint32_t)(hi >> (b - 64)) & 0x3FFu;
    return (uint32_t)((lo >> b) | (hi << (64 - b))) & 0x3FFu;
}

// expand one 10x10 game into 144 Tile.value bytes (dst 4-byte aligned; shared or global memory).  CODES: render slide tiles as
// 5/6 (export); the observation tables map slide tiles to the body values, so the encode path skips that.
template <bool SLIDE, bool CODES>
__device__ __forceinline__ void expand_tile10(const BitCells<SLIDE, 10>& g, int r1, int c1, int r2, int c2, int8_t* dst) {
    uint32_t* w = (uint32_t*)dst;
    w[0] = w[1] = w[2] = 0xFFFFFFFFu;  // border rows: WALL = -1
    w[33] = w[34] = w[35] = 0xFFFFFFFFu;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t occ = row_bits10(g.occ_lo, g.occ_hi, r), own = row_bits10(g.own_lo, g.own_hi, r);
        const uint32_t sld = (SLIDE && CODES) ? row_bits10(g.sld_lo, g.sld_hi, r) : 0u;
        w[3 * (r + 1) + 0] = tiles4<SLIDE && CODES>(occ << 1, own << 1, sld << 1) | 0x000000FFu;          // [wall, i0, i1, i2]
        w[3 * (r + 1) + 1] = tiles4<SLIDE && CODES>(occ >> 3, own >> 3, sld >> 3);                         // [i3 .. i6]
        w[3 * (r + 1) + 2] = tiles4<SLIDE && CODES>((occ >> 7) & 7u, own >> 7, sld >> 7) | 0xFF000000u;   // [i7, i8, i9, wall]
    }
    // heads overlay, P2 second so it wins a shared cell (reference game.py:205-214); positions may sit on the border
    dst[(r1 + 1) * 12 + c1 + 1] = TRON_TILE_P1_HEAD;
    dst[(r2 + 1) * 12 + c2 + 1] = TRON_TILE_P2_HEAD;
}
// any W*H <= 128: byte by byte
template <bool SLIDE>
__device__ __forceinline__ void expand_tile_generic(const BitCells<SLIDE, 0>& g, int r1, int c1, int r2, int c2, int8_t* dst) {
    const int W = g.Wr, H = g.Hr, Hc = H + 2;
    for (int c = 0; c < Hc; ++c) { dst[c] = TRON_TILE_WALL; dst[(W + 1) * Hc + c] = TRON_TILE_WALL; }
    for (int r = 0; r < W; ++r) {
        int8_t* row = dst + (r + 1) * Hc;
        row[0] = TRON_TILE_WALL; row[H + 1] = TRON_TILE_WALL;
        for (int c = 0; c < H; ++c) {
            const int b = r * H + c;
            const unsigned long long o = b < 64 ? g.occ_lo : g.occ_hi, v = b < 64 ? g.own_lo : g.own_hi, s = b < 64 ? g.sld_lo : g.sld_hi;
            const int occ = (int)((o >> (b & 63)) & 1ull), own = (int)((v >> (b & 63)) & 1ull), sl = SLIDE ? (int)((s >> (b & 63)) & 1ull) : 0;
            row[c + 1] = (int8_t)(occ ? (sl ? (own ? TRON_TILE_P2_SLIDE : TRON_TILE_P1_SLIDE) : (own ? TRON_TILE_P2_BODY : TRON_TILE_P1_BODY)) : TRON_TILE_EMPTY);
        }
    }
    dst[(r1 + 1) * Hc + c1 + 1] = TRON_TILE_P1_HEAD;
    dst[(r2 + 1) * Hc + c2 + 1] = TRON_TILE_P2_HEAD;
}
template <bool SLIDE, int W_T, bool CODES>
__device__ __forceinline__ void expand_tile(const BitCells<SLIDE, W_T>& g, int r1, int c1, int r2, int c2, int8_t* dst) {
    if constexpr (W_T == 10) expand_tile10<SLIDE, CODES>(g, r1, c1, r2, c2, dst);
    else expand_tile_generic<SLIDE>(g, r1, c1, r2, c2, dst);
}

// ------------------------------------------------------------------------------------------------ observation delta
// tron_step_args.obs_prev: `obs` already holds the observation of every game's pre-tick state, so only the 32-byte units whose
// cells this tick changes are written.  A unit holds 16 cells (bf16) or 8 (f32) of one plane, so unit boundaries fall on plane
// boundaries and one unit-in-plane mask per game serves all its lut planes.  int8 planes (144 B) straddle units: full rows.
constexpr int kDeltaUnit = 32;  // bytes; a full L2 sector, so no partial-sector write reaches HBM
template <int W_T, int OD, int LP, int MODE>
struct DeltaObs {
    static constexpr int ES = OD == TRON_F32 ? 4 : OD == TRON_BF16 ? 2 : 1;
    static constexpr bool kOn = W_T == 10 && MODE == MODE_STEP && LP > 0 && OD != TRON_I8;
    static constexpr int CPU = kDeltaUnit / ES;       // cells per unit: 16 (bf16), 8 (f32)
    static constexpr int UPP = 144 / CPU;             // units per plane: 9, 18
    static constexpr int CHU = kDeltaUnit / 16;       // 16-byte chunks per unit
};
__device__ __forceinline__ int head_cell10(int r, int c) {
    const int h = (r + 1) * 12 + c + 1;
    return TRON_DCHECK(h >= 0 && h < 144, DBG_CELL_INDEX) ? h : 0;
}
// bit u set: unit u of the lut planes holds an interior cell whose occ or own bit changed (d_lo / d_hi).  The caller adds the
// cells of heads that moved: a head cell shows the head tile whatever its planes say, and may lie on the border ring.
template <int CPU>
__device__ __forceinline__ uint32_t dirty_units10(unsigned long long d_lo, unsigned long long d_hi) {
    unsigned long long c[3] = {0ull, 0ull, 0ull};  // cell bits of the 12x12 tile
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned long long d = row_bits10(d_lo, d_hi, r);
        const int s = (r + 1) * 12 + 1, w = s >> 6, o = s & 63;
        c[w] |= d << o;
        if (o + 10 > 64) c[w + 1] |= d >> (64 - o);
    }
    uint32_t um = 0;
#pragma unroll
    for (int u = 0; u < 144 / CPU; ++u) {
        const int b = u * CPU;
        um |= (((c[b >> 6] >> (b & 63)) & ((1ull << CPU) - 1ull)) != 0ull ? 1u : 0u) << u;
    }
    return um;
}
// CTA-wide exclusive scan of one count per thread (kBitsThreads threads); returns this thread's offset, *total = the sum
__device__ __forceinline__ int cta_exclusive_scan(int n, int* wsum, int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    int base = 0, sum = 0;
#pragma unroll
    for (int w = 0; w < kBitsThreads / 32; ++w) {
        base += w < warp ? wsum[w] : 0;
        sum += wsum[w];
    }
    *total = sum;
    return base + incl - n;
}

// ------------------------------------------------------------------------------------------------ the kernel
// DELTA: the obs_prev instantiation (single tick, changed units only); every other launch runs DELTA = false, whose code is the
// full-row kernel unchanged
template <bool SLIDE, int W_T, int OD, int LP, bool CP, int CH, int MODE, bool DELTA>
__global__ void __launch_bounds__(kBitsThreads) step_bits_kernel(const StepParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int C = W_T ? (W_T + 2) * (W_T + 2) : p.C;
    int8_t* tile = (int8_t*)smem_raw;  // [G][C] Tile.value bytes, only a staging area for the encode
    uint8_t* tflag = (uint8_t*)(tile + ((p.G * C + 15) & ~15));  // [G] "this game just finished" (terminal-frame pass)
    PlaneTab* smtab = (PlaneTab*)(tflag + ((p.G + 15) & ~15));   // [2][3] tables for the linear schedule
    using DO = DeltaObs<W_T, OD, LP, MODE>;
    constexpr bool delta = DELTA && DO::kOn;
    int* wsum = (int*)(smtab + 6);                               // [4] warp sums of the dirty-unit scan
    uint16_t* dlist = (uint16_t*)(wsum + 4);                     // [<= G * 2P * UPP] game << 8 | unit of the game's row
    const int tid = threadIdx.x;
    // store schedule: linear (one contiguous 512-byte run per warp store) on the 10x10 board; TRON_OPT_ENCODE_VARIANT 8 selects the
    // per-plane schedule of encode_tile() for comparison
    const bool linear = W_T == 10 && !(p.variant & 8);
    const bool linear4 = W_T == 0 && LP == 3 && (C & 3) == 0 && C <= 256 && !(p.variant & 8);  // other boards, pop_up planes: units of 4 cells (step_kernels.cuh)
    if (LP > 0 && (linear || linear4)) {
        if (tid < 6) smtab[tid] = p.tab[tid / 3][tid % 3];
        __syncthreads();
    }
    using Cells = BitCells<SLIDE, W_T>;
    const long long env0 = (long long)blockIdx.x * p.G;
    const int nG = (int)min((long long)p.G, (long long)p.N - env0);
    const bool owner = tid < nG;
    const long long env = env0 + tid;
    Cells g;
    g.clear(); g.Wr = p.W; g.Hr = p.H;
    EnvState e = unpack_meta(make_uint2(0, 0));
    if (owner) {
        if (!(MODE == MODE_RESET && p.env_mask == nullptr)) set_planes(g, load_planes<SLIDE>(p, env));
        e = unpack_meta(p.meta[env]);
    }
    const int T = MODE == MODE_STEP ? p.T : 1;
    for (int t = 0; t < T; ++t) {
        bool fin = false;
        // pre-tick observation inputs (delta path): occ / own words and head cells
        const unsigned long long occ0_lo = g.occ_lo, occ0_hi = g.occ_hi, own0_lo = g.own_lo, own0_hi = g.own_hi;
        const int hp1 = delta ? head_cell10(e.r1, e.c1) : 0, hp2 = delta ? head_cell10(e.r2, e.c2) : 0;
        if (MODE != MODE_OBSERVE && owner) {
            BoxRegs bx;
            fin = env_tick<MODE, false, (SLIDE ? FEAT_ALL : FEAT_EPS)>(g, p, e, env, t, tid, bx);  // BITS10 has no slide plane
        }
        if constexpr (LP > 0 && MODE == MODE_STEP) {
            if (p.obs_term) {  // last frame of the games that just finished (-> obs_terminal)
                if (owner) {
                    tflag[tid] = fin ? 1 : 0;
                    if (fin) expand_tile<SLIDE, W_T, false>(g, e.tr1, e.tc1, e.tr2, e.tc2, tile + tid * C);
                }
                __syncthreads();
                const int tt = p.obs_every_tick ? t : 0;
                if (linear) encode_tile_linear144<kBitsThreads, OD, LP, CP>(tile, nG, env0, p, tt, smtab, p.obs_term, tflag);
                else if (linear4) encode_tile_linear4<kBitsThreads, OD, LP, CP>(tile, C, nG, env0, p, tt, smtab, p.obs_term, tflag);
                else encode_tile<(W_T == 10 ? 144 : 0), kBitsThreads, OD, LP, CP, CH>(tile, nG, env0, p, tt, p.obs_term, tflag);
                __syncthreads();
            }
        }
        if (fin) g.clear();
        if (MODE == MODE_OBSERVE && owner) emit_extra(p, env);
        if constexpr (LP > 0) {
            if (MODE == MODE_OBSERVE || p.obs_every_tick || t == T - 1) {
                if (owner) expand_tile<SLIDE, W_T, false>(g, e.r1, e.c1, e.r2, e.c2, tile + tid * C);
                if constexpr (delta) {
                    {  // T == 1: list the CTA's changed units in row order, then encode and store only those
                        constexpr int P = Linear144<OD, LP, CP>::P, CPG = Linear144<OD, LP, CP>::CPG;
                        int n = 0;
                        uint32_t um = 0;
                        if (owner) {
                            const int hn1 = head_cell10(e.r1, e.c1), hn2 = head_cell10(e.r2, e.c2);
                            um = dirty_units10<DO::CPU>((occ0_lo ^ g.occ_lo) | (own0_lo ^ g.own_lo), (occ0_hi ^ g.occ_hi) | (own0_hi ^ g.own_hi));
                            if (hn1 != hp1) um |= (1u << (hp1 / DO::CPU)) | (1u << (hn1 / DO::CPU));
                            if (hn2 != hp2) um |= (1u << (hp2 / DO::CPU)) | (1u << (hn2 / DO::CPU));
                            n = __popc(um) * 2 * LP;  // the constant plane never changes
                        }
                        int total;
                        int off = cta_exclusive_scan(n, wsum, &total);
                        if (owner) {
#pragma unroll
                            for (int pq = 0; pq < 2 * P; ++pq) {
                                if (CP && pq % P == LP) continue;
                                for (uint32_t m = um; m; m &= m - 1u) {
                                    if (TRON_DCHECK(off < p.G * 2 * LP * DO::UPP, DBG_OBS_UNIT))
                                        dlist[off] = (uint16_t)((tid << 8) | (pq * DO::UPP + __ffs(m) - 1));
                                    ++off;
                                }
                            }
                        }
                        __syncthreads();
                        uint4* obase = (uint4*)p.obs + (size_t)env0 * CPG;
                        for (int i = tid; i < total * DO::CHU; i += kBitsThreads) {
                            const int k = i / DO::CHU;
                            const uint32_t ent = dlist[k];
                            const int ge = (int)(ent >> 8), j = (int)(ent & 0xFFu) * DO::CHU + (i - k * DO::CHU);
                            if (!TRON_DCHECK(ge < nG && j < CPG, DBG_OBS_UNIT)) continue;
                            st_cs(obase + (size_t)ge * CPG + j, encode_chunk144<OD, LP, CP>(tile, ge, j, p, smtab));
                        }
                        continue;  // T == 1: nothing follows in this tick
                    }
                }
                __syncthreads();
                const int tt = (MODE == MODE_STEP && p.obs_every_tick) ? t : 0;
                if (linear) encode_tile_linear144<kBitsThreads, OD, LP, CP>(tile, nG, env0, p, tt, smtab);
                else if (linear4) encode_tile_linear4<kBitsThreads, OD, LP, CP>(tile, C, nG, env0, p, tt, smtab);
                else encode_tile<(W_T == 10 ? 144 : 0), kBitsThreads, OD, LP, CP, CH>(tile, nG, env0, p, tt);
                if (T > 1) __syncthreads();  // the tile is rewritten by the next tick
            }
        }
    }
    if (MODE != MODE_OBSERVE && owner) {
        store_planes(p, env, g);
        p.meta[env] = pack_meta(e);
    }
}

// ------------------------------------------------------------------------------------------------ launch
static size_t bits_smem(int G, int C, int LP) {
    if (LP == 0) return 0;
    return (size_t)((G * C + 15) & ~15) + (size_t)((G + 15) & ~15) + 6 * sizeof(PlaneTab);
}

template <bool SLIDE, int W_T, int OD, int LP, bool CP, int CH, int MODE>
static int launch_bits_one(const StepParams& p_in, cudaStream_t s) {
    using DO = DeltaObs<W_T, OD, LP, MODE>;
    StepParams p = p_in;
    // the delta store covers single ticks of the linear schedule; TRON_OPT_ENCODE_VARIANT 64 forces full rows (A/B timing)
    if (!DO::kOn || p.T != 1 || (p.variant & (8 | 64))) p.obs_prev = 0;
    const long long n_tiles = ((long long)p.N + p.G - 1) / p.G;
    size_t smem = bits_smem(p.G, p.C, LP);
    if (p.obs_prev) smem += 4 * sizeof(int) + (size_t)p.G * 2 * LP * DO::UPP * sizeof(uint16_t);
    if (LP > 0 && MODE == MODE_STEP && n_tiles > 8ll * sm_count()) {
        // Cap the resident CTAs per SM by padding the dynamic shared memory: floor(228 KB / (smem + 1 KB reserved)) == cap.  The fused
        // kernels are write streams; with fewer of them per SM than the register limit (8) the DRAM pages see longer bursts
        // (measured: 4 is best for the two-plane kernels, 5 with the slide plane whose tick phase is longer).
        // int8 planes move fewer bytes per CTA: one plane stays uncapped (0.92; 0.78 at 4), three / four planes take 5 (0.985).
        // The delta store writes about a third of the bytes per CTA: 5 (headline 0.361 ms at 4, 0.320 at 5, 0.340 at 6 per tick,
        // profiles/r3_obs_delta.jsonl).
        const long long cap = g_bits_ctas_per_sm > 0 ? g_bits_ctas_per_sm : (OD == TRON_I8 ? (LP == 1 ? 32 : 5) : (SLIDE || p.obs_prev) ? 5 : 4);
        const size_t want = (size_t)(228 * 1024) / (size_t)(cap + 1) - 1024 + 256;
        if (want > smem && want <= 200 * 1024) smem = want;
    }
    auto kern = step_bits_kernel<SLIDE, W_T, OD, LP, CP, CH, MODE, false>;
    if constexpr (DO::kOn) {
        if (p.obs_prev) kern = step_bits_kernel<SLIDE, W_T, OD, LP, CP, CH, MODE, true>;
    }
    if (smem > 48 * 1024 && ensure_dynamic_smem((const void*)kern, smem) != TRON_OK) return TRON_ERR_CUDA;
    kern<<<(unsigned)n_tiles, kBitsThreads, smem, s>>>(p);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}
template <bool SLIDE, int W_T, int OD, int CH, int MODE>
static int launch_bits_enc(const StepParams& p, int enc_kind, cudaStream_t s) {
    switch (enc_kind) {
        case 1: return launch_bits_one<SLIDE, W_T, OD, 1, false, CH, MODE>(p, s);
        case 2: return launch_bits_one<SLIDE, W_T, OD, 3, false, CH, MODE>(p, s);
        case 3: return launch_bits_one<SLIDE, W_T, OD, 3, true, CH, MODE>(p, s);
        default: return TRON_ERR_INVALID;
    }
}
// CH8: cells per encode item of the non-f32 dtypes (8 when C % 8 == 0, else 4 or 1); f32 uses min(CH8, 4) (whole-sector stores)
template <bool SLIDE, int W_T, int CH8>
static int launch_bits_geo(const StepParams& p, int mode, int od, int enc_kind, cudaStream_t s) {
    constexpr int CH32 = CH8 == 8 ? 4 : CH8;
    if (mode == MODE_RESET) return launch_bits_one<SLIDE, W_T, TRON_I8, 0, false, CH8, MODE_RESET>(p, s);
    if (mode == MODE_STEP && enc_kind == 0) return launch_bits_one<SLIDE, W_T, TRON_I8, 0, false, CH8, MODE_STEP>(p, s);
    if (mode == MODE_STEP) {
        if (od == TRON_BF16) return launch_bits_enc<SLIDE, W_T, TRON_BF16, CH8, MODE_STEP>(p, enc_kind, s);
        if (od == TRON_F32) return launch_bits_enc<SLIDE, W_T, TRON_F32, CH32, MODE_STEP>(p, enc_kind, s);
        if (od == TRON_I8) return launch_bits_enc<SLIDE, W_T, TRON_I8, CH8, MODE_STEP>(p, enc_kind, s);
    } else if (mode == MODE_OBSERVE) {
        if (od == TRON_BF16) return launch_bits_enc<SLIDE, W_T, TRON_BF16, CH8, MODE_OBSERVE>(p, enc_kind, s);
        if (od == TRON_F32) return launch_bits_enc<SLIDE, W_T, TRON_F32, CH32, MODE_OBSERVE>(p, enc_kind, s);
        if (od == TRON_I8) return launch_bits_enc<SLIDE, W_T, TRON_I8, CH8, MODE_OBSERVE>(p, enc_kind, s);
    }
    return TRON_ERR_INVALID;
}

int launch_step_bits10(const StepParams& p_in, int mode, int od, int enc_kind, cudaStream_t s) {
    StepParams p = p_in;
    p.G = tile_envs_small_grid(p.N);
    return launch_bits_geo<false, 10, 8>(p, mode, od, enc_kind, s);
}
int launch_step_bits(const StepParams& p_in, int mode, int od, int enc_kind, cudaStream_t s) {
    StepParams p = p_in;
    if (p.W == 10 && p.H == 10) {
        p.G = tile_envs_small_grid(p.N);
        return launch_bits_geo<true, 10, 8>(p, mode, od, enc_kind, s);
    }
    int g = 18432 / p.C;  // games per CTA: ~18 KB of staging, a multiple of 16 so the tile stays 16-byte aligned
    g -= g % 16;
    g = g < 16 ? 16 : (g > kBitsThreads ? kBitsThreads : g);
    const int small = tile_envs_small_grid(p.N);
    p.G = small < g ? small : g;
    if (p.C % 4 == 0) return launch_bits_geo<true, 0, 4>(p, mode, od, enc_kind, s);
    return launch_bits_geo<true, 0, 1>(p, mode, od, enc_kind, s);
}

// ------------------------------------------------------------------------------------------------ export / import
template <bool SLIDE, int W_T>
__global__ void bits_export_kernel(const StepParams p, const uint2* __restrict__ meta, int8_t* tiles) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.N) return;
    BitCells<SLIDE, W_T> g;
    g.clear(); g.Wr = p.W; g.Hr = p.H;
    set_planes(g, load_planes<SLIDE>(p, env));
    const EnvState e = unpack_meta(meta[env]);
    expand_tile<SLIDE, W_T, true>(g, e.r1, e.c1, e.r2, e.c2, tiles + (size_t)env * p.C);
}
// tiles -> planes: trail tiles set bits (BITS10 stores slide tiles as bodies), everything else is implicit
template <bool SLIDE, int W_T>
__global__ void bits_import_kernel(const StepParams p, const int8_t* __restrict__ tiles, bool derive_heads) {
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.N) return;
    BitCells<SLIDE, W_T> g;
    g.clear(); g.Wr = p.W; g.Hr = p.H;
    const int8_t* t = tiles + (size_t)env * p.C;
    for (int r = 0; r < p.W; ++r)
        for (int c = 0; c < p.H; ++c) {
            const int v = t[(r + 1) * p.Hc + c + 1];
            if (v == TRON_TILE_P1_BODY || v == TRON_TILE_P2_BODY) g.put(r, c, v);
            else if (v == TRON_TILE_P1_SLIDE) g.put(r, c, SLIDE ? (int)TRON_TILE_P1_SLIDE : (int)TRON_TILE_P1_BODY);
            else if (v == TRON_TILE_P2_SLIDE) g.put(r, c, SLIDE ? (int)TRON_TILE_P2_SLIDE : (int)TRON_TILE_P2_BODY);
        }
    store_planes(p, env, g);
    uint32_t packed;
    if (derive_heads && heads_from_tiles(t, p.W, p.H, packed)) p.meta[env].x = packed;  // the bit planes cannot hold heads: they go into the meta
}
int launch_bits_export(const StepParams& p, const void* meta, int8_t* tiles, cudaStream_t s) {
    const unsigned grid = (unsigned)((p.N + 127) / 128);
    if (p.layout == TRON_LAYOUT_BITS10) bits_export_kernel<false, 10><<<grid, 128, 0, s>>>(p, (const uint2*)meta, tiles);
    else if (p.W == 10 && p.H == 10) bits_export_kernel<true, 10><<<grid, 128, 0, s>>>(p, (const uint2*)meta, tiles);
    else bits_export_kernel<true, 0><<<grid, 128, 0, s>>>(p, (const uint2*)meta, tiles);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}
int launch_bits_import(const StepParams& p, const int8_t* tiles, bool derive_heads, cudaStream_t s) {
    const unsigned grid = (unsigned)((p.N + 127) / 128);
    if (p.layout == TRON_LAYOUT_BITS10) bits_import_kernel<false, 10><<<grid, 128, 0, s>>>(p, tiles, derive_heads);
    else if (p.W == 10 && p.H == 10) bits_import_kernel<true, 10><<<grid, 128, 0, s>>>(p, tiles, derive_heads);
    else bits_import_kernel<true, 0><<<grid, 128, 0, s>>>(p, tiles, derive_heads);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

}  // namespace tron
