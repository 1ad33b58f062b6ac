// step_kernels.cuh -- the fused TRON tick: move, collision, winner/draw, trail write, auto-reset,
// reward and observation encoding for a tile of G consecutive games per CTA.
//
// Data flow per CTA (one tile = G games x C cells of int8 Tile.value, contiguous in HBM):
//   1. one elected thread pulls the whole tile into shared memory with a 1-D bulk (TMA-engine) copy
//      completing on an mbarrier, while the other threads fetch per-game metadata and actions;
//   2. thread-per-game runs the reference's tick on its game's cells in shared memory
//      (reference tron/game.py:149-277), emits reward/done/winner, decides auto-reset + spawn;
//   3. all threads rebuild reset games from a per-CTA template grid;
//   4. the final tile goes back to HBM as one bulk store while all threads encode both players'
//      observation planes straight from shared memory with 16-byte streaming stores (PRMT byte-LUT).
// HBM traffic per game-tick: C read + C written (grid) + 2*P*C*sizeof(obs) written + ~30 B metadata.
#pragma once
#include "common.cuh"
#include "tick_core.cuh"

namespace tron {

// ---- observation element packing --------------------------------------------------------------
// 4 cells -> 4 encoded elements of dtype OD, returned as raw 32-bit words (1 word i8, 2 bf16, 4 f32)
template <int OD>
struct Enc4;
template <>
struct Enc4<TRON_BF16> {
    static constexpr int WORDS = 2;
    __device__ __forceinline__ static void run(const PlaneTab& t, uint32_t sel, uint32_t* o) {
        const uint32_t lo = lut4(t.lo0, t.lo1, sel), hi = lut4(t.hi0, t.hi1, sel);
        o[0] = __byte_perm(lo, hi, 0x5140);
        o[1] = __byte_perm(lo, hi, 0x7362);
    }
    __device__ __forceinline__ static void fill(float v, uint32_t* o) {
        const uint32_t b = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v));
        o[0] = o[1] = b | (b << 16);
    }
};
template <>
struct Enc4<TRON_F32> {
    static constexpr int WORDS = 4;
    __device__ __forceinline__ static void run(const PlaneTab& t, uint32_t sel, uint32_t* o) {
        const uint32_t lo = lut4(t.lo0, t.lo1, sel), hi = lut4(t.hi0, t.hi1, sel);
        o[0] = __byte_perm(lo, hi, 0x4044) & 0xFFFF0000u;  // bytes: [x, x, lo0, hi0] -> keep upper half
        o[1] = __byte_perm(lo, hi, 0x5144) & 0xFFFF0000u;
        o[2] = __byte_perm(lo, hi, 0x6244) & 0xFFFF0000u;
        o[3] = __byte_perm(lo, hi, 0x7344) & 0xFFFF0000u;
    }
    __device__ __forceinline__ static void fill(float v, uint32_t* o) { o[0] = o[1] = o[2] = o[3] = __float_as_uint(v); }
};
template <>
struct Enc4<TRON_I8> {
    static constexpr int WORDS = 1;
    __device__ __forceinline__ static void run(const PlaneTab& t, uint32_t sel, uint32_t* o) { o[0] = lut4(t.lo0, t.lo1, sel); }
    __device__ __forceinline__ static void fill(float v, uint32_t* o) {
        const uint32_t b = (uint32_t)(uint8_t)(int8_t)v;
        o[0] = b * 0x01010101u;
    }
};

template <int OD>
__device__ __forceinline__ int elem_size() { return OD == TRON_F32 ? 4 : OD == TRON_BF16 ? 2 : 1; }

// Encode both players' observation planes of a tile of nG games held in shared memory as int8 Tile.values.
// Every warp-wide store covers whole 32-byte sectors; values come from 8-entry byte tables via PRMT (common.cuh).
// `only` != nullptr: encode just the games whose flag is set (terminal frames of finished games -> obs_terminal).
template <int C_T, int NT, int OD, int LP, bool CP, int CH>
__device__ __forceinline__ void encode_tile(const int8_t* tile, int nG, long long env0, const StepParams& p, int t, void* out = nullptr,
                                            const uint8_t* only = nullptr) {
    const int C = C_T ? C_T : p.C;
    const int tid = threadIdx.x;
            constexpr int ES = OD == TRON_F32 ? 4 : OD == TRON_BF16 ? 2 : 1;
            const int P = p.P;
            const size_t tick_off = (size_t)t * (size_t)p.N * 2 * (size_t)P * (size_t)C * ES;
            char* obase = (char*)(out ? out : p.obs) + tick_off;
            if constexpr (CH >= 4) {
                const int per = C / CH;
                // one item = CH consecutive cells of one game -> one store per (player, plane)
                auto emit = [&](int e, int ch) {
                    const int8_t* cells = tile + e * C + ch * CH;
                    uint32_t sel[CH / 4];
                    if constexpr (CH == 8) { const uint2 w = *(const uint2*)cells; sel[0] = cell_selector(w.x); sel[1] = cell_selector(w.y); }
                    else { sel[0] = cell_selector(*(const uint32_t*)cells); }
                    char* row0 = obase + ((size_t)(env0 + e) * 2 * P * C + (size_t)ch * CH) * ES;
#pragma unroll
                    for (int pl = 0; pl < 2; ++pl) {
#pragma unroll
                        for (int q = 0; q < LP + (CP ? 1 : 0); ++q) {
                            uint32_t o[(CH / 4) * Enc4<OD>::WORDS];
#pragma unroll
                            for (int h = 0; h < CH / 4; ++h) {
                                if (q < LP) Enc4<OD>::run(p.tab[pl][q < LP ? q : 0], sel[h], o + h * Enc4<OD>::WORDS);
                                else Enc4<OD>::fill(p.const_plane, o + h * Enc4<OD>::WORDS);
                            }
                            char* dst = row0 + (size_t)(pl * P + q) * C * ES;
                            constexpr int NW = (CH / 4) * Enc4<OD>::WORDS;
                            if (NW == 8) { st_cs((uint4*)dst, make_uint4(o[0], o[1], o[2], o[3])); st_cs((uint4*)dst + 1, make_uint4(o[4 % NW], o[5 % NW], o[6 % NW], o[7 % NW])); }
                            else if (NW == 4) st_cs((uint4*)dst, make_uint4(o[0], o[1 % NW], o[2 % NW], o[3 % NW]));
                            else if (NW == 2) st_cs((uint2*)dst, make_uint2(o[0], o[1 % NW]));
                            else *(uint32_t*)dst = o[0];
                        }
                    }
                };
                if (C_T == 0 && per >= 4 * NT) {  // large grids: game-major loops, no per-item division
                    for (int e = 0; e < nG; ++e) {
                        if (only && !only[e]) continue;
                        for (int ch = tid; ch < per; ch += NT) emit(e, ch);
                    }
                } else {
                    for (int it = tid; it < nG * per; it += NT) {
                        const int e = it / per;
                        if (only && !only[e]) continue;
                        emit(e, it - e * per);
                    }
                }
            } else {  // scalar fallback for odd cell counts
                for (int it = tid; it < nG * C; it += NT) {
                    const int e = it / C, c = it - e * C;
                    if (only && !only[e]) continue;
                    const uint32_t sel = (uint32_t)tile[it] & 7u;
                    for (int pl = 0; pl < 2; ++pl)
                        for (int q = 0; q < LP + (CP ? 1 : 0); ++q) {
                            uint32_t o[Enc4<OD>::WORDS];
                            if (q < LP) Enc4<OD>::run(p.tab[pl][q < LP ? q : 0], sel, o); else Enc4<OD>::fill(p.const_plane, o);
                            char* dst = obase + ((size_t)((env0 + e) * 2 + pl) * P + q) * C * ES + (size_t)c * ES;
                            if (ES == 4) *(uint32_t*)dst = o[0];
                            else if (ES == 2) *(uint16_t*)dst = (uint16_t)o[0];
                            else *(uint8_t*)dst = (uint8_t)o[0];
                        }
                }
            }
        }

// ---- linear encode schedule (10x10 boards) ---------------------------------------------------------
// The observation of one game is one contiguous run of 2*P planes; here item j of a game is its j-th 16-byte chunk, whatever
// plane it falls into, so every warp-wide store is ONE contiguous 512-byte run (encode_tile() instead issues one store per
// (player, plane) whose lanes follow the cells, i.e. 2*P interleaved runs of 288 B).  Costs a selector recomputation per chunk.
template <int OD, int LP, bool CP>
struct Linear144 {
    static constexpr int C = 144, ES = OD == TRON_F32 ? 4 : OD == TRON_BF16 ? 2 : 1, P = (LP + (CP ? 1 : 0)) > 0 ? LP + (CP ? 1 : 0) : 1;
    static constexpr int CPC = 16 / ES;           // cells per 16-byte chunk: 8 (bf16), 4 (f32), 16 (i8)
    static constexpr int CPP = C / CPC;           // chunks per plane: 18, 36, 9
    static constexpr int CPG = 2 * P * CPP;       // chunks per game
};
// chunk j of game e of the tile (both players' planes in row order)
template <int OD, int LP, bool CP>
__device__ __forceinline__ uint4 encode_chunk144(const int8_t* tile, int e, int j, const StepParams& p, const PlaneTab* smtab) {
    using L = Linear144<OD, LP, CP>;
    const int pq = j / L::CPP, ch = j - pq * L::CPP, pl = pq / L::P, q = pq - pl * L::P;
    uint32_t o[4];
    if (CP && q == LP) {
        uint32_t f[Enc4<OD>::WORDS];
        Enc4<OD>::fill(p.const_plane, f);
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k] = f[k % Enc4<OD>::WORDS];
    } else {
        const PlaneTab tb = smtab[pl * 3 + q];
        const int8_t* cells = tile + e * L::C + ch * L::CPC;
        if constexpr (L::CPC == 8) {
            const uint2 w = *(const uint2*)cells;
            Enc4<OD>::run(tb, cell_selector(w.x), o); Enc4<OD>::run(tb, cell_selector(w.y), o + 2);
        } else if constexpr (L::CPC == 4) {
            Enc4<OD>::run(tb, cell_selector(*(const uint32_t*)cells), o);
        } else {
            const uint4 w = *(const uint4*)cells;
            Enc4<OD>::run(tb, cell_selector(w.x), o); Enc4<OD>::run(tb, cell_selector(w.y), o + 1);
            Enc4<OD>::run(tb, cell_selector(w.z), o + 2); Enc4<OD>::run(tb, cell_selector(w.w), o + 3);
        }
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
}
template <int NT, int OD, int LP, bool CP>
__device__ __forceinline__ void encode_tile_linear144(const int8_t* tile, int nG, long long env0, const StepParams& p, int t, const PlaneTab* smtab,
                                                      void* out = nullptr, const uint8_t* only = nullptr) {
    constexpr int CPG = Linear144<OD, LP, CP>::CPG;
    const size_t tick_off = (size_t)t * (size_t)p.N * CPG * 16;
    uint4* obase = (uint4*)((char*)(out ? out : p.obs) + tick_off) + (size_t)env0 * CPG;
    for (int it = threadIdx.x; it < nG * CPG; it += NT) {
        const int e = it / CPG, j = it - e * CPG;
        if (only && !only[e]) continue;
        st_cs(obase + it, encode_chunk144<OD, LP, CP>(tile, e, j, p, smtab));
    }
}

// The same linear schedule for any board with C % 4 == 0, in units of 4 cells (4 / 8 / 16 bytes for i8 / bf16 / f32): consecutive
// lanes write consecutive units of the batch's contiguous observation rows across plane, player and game boundaries, so a warp
// store is one contiguous run (encode_tile() leaves a partial sector at every 2*C*ES-byte plane end: 8x8 boards ran at 0.73).
// div_* are exact magic divisions for the small ranges involved (n < 2^20, d < 2^12).
__device__ __forceinline__ uint32_t magic_of(uint32_t d) { return 0xFFFFFFFFu / d + 1u; }
__device__ __forceinline__ int magic_div(int n, uint32_t magic, int d) { return d == 1 ? n : (int)__umulhi((uint32_t)n, magic); }
template <int NT, int OD, int LP, bool CP>
__device__ __forceinline__ void encode_tile_linear4(const int8_t* tile, int C, int nG, long long env0, const StepParams& p, int t, const PlaneTab* smtab,
                                                    void* out = nullptr, const uint8_t* only = nullptr) {
    constexpr int ES = OD == TRON_F32 ? 4 : OD == TRON_BF16 ? 2 : 1, P = (LP + (CP ? 1 : 0)) > 0 ? LP + (CP ? 1 : 0) : 1;
    constexpr int UB = 4 * ES;                     // bytes per unit
    const int UPP = C >> 2, UPG = 2 * P * UPP;     // units per plane / per game
    const uint32_t m_upg = magic_of((uint32_t)UPG), m_upp = magic_of((uint32_t)UPP);
    char* obase = (char*)(out ? out : p.obs) + ((size_t)t * (size_t)p.N + (size_t)env0) * (size_t)UPG * UB;
    for (int it = threadIdx.x; it < nG * UPG; it += NT) {
        const int e = magic_div(it, m_upg, UPG), j = it - e * UPG;
        if (only && !only[e]) continue;
        const int pq = magic_div(j, m_upp, UPP), ch = j - pq * UPP, pl = pq >= P ? 1 : 0, q = pq - pl * P;
        uint32_t o[Enc4<OD>::WORDS];
        if (CP && q == LP) Enc4<OD>::fill(p.const_plane, o);
        else Enc4<OD>::run(smtab[pl * 3 + q], cell_selector(*(const uint32_t*)(tile + e * C + ch * 4)), o);
        char* dst = obase + (size_t)it * UB;
        if constexpr (Enc4<OD>::WORDS == 4) st_cs((uint4*)dst, make_uint4(o[0], o[1 % Enc4<OD>::WORDS], o[2 % Enc4<OD>::WORDS], o[3 % Enc4<OD>::WORDS]));
        else if constexpr (Enc4<OD>::WORDS == 2) st_cs((uint2*)dst, make_uint2(o[0], o[1 % Enc4<OD>::WORDS]));
        else *(uint32_t*)dst = o[0];
    }
}

// ---- the kernel -----------------------------------------------------------------------------
// C_T: cells per env at compile time (0 = runtime), NT threads, OD obs dtype, LP lut planes (0 = no obs),
// CP const plane, CH cells per encode item (8, 4 or 1; C % CH == 0), MODE.
template <int C_T, int NT, int OD, int LP, bool CP, int CH, int MODE>
__global__ void __launch_bounds__(NT) step_tile_kernel(const StepParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int C = C_T ? C_T : p.C;
    const int G = p.G;
    const int tid = threadIdx.x;
    const long long env0 = (long long)blockIdx.x * G;
    const int nG = (int)min((long long)G, (long long)p.N - env0);

    // shared layout: tile[G*C] | template[C] (16B padded) | hidx[G] (ushort2) | rflag[G] | mbarrier
    int8_t* tile = (int8_t*)smem_raw;
    const int tile_bytes_full = (G * C + 15) & ~15;
    int8_t* tmpl = tile + tile_bytes_full;
    ushort2* hidx = (ushort2*)(tmpl + ((C + 15) & ~15));
    uint8_t* rflag = (uint8_t*)(hidx + G);
    uint64_t* bar = (uint64_t*)(((uintptr_t)(rflag + G) + 7) & ~(uintptr_t)7);
    PlaneTab* smtab = (PlaneTab*)(((uintptr_t)(bar + 1) + 15) & ~(uintptr_t)15);  // [2][3] tables of the linear schedule (10x10 only)
    constexpr bool kLinear = C_T == 144 && LP > 0;
    // other small boards with pop_up planes: the unit-of-4-cells linear schedule (measured at 8x8: pop_up 0.79 -> 0.86; one-plane
    // encodings and boards from 12x12 up are faster with the per-plane schedule, whose stores are twice as wide)
    const bool linear4 = C_T == 0 && LP == 3 && (C & 3) == 0 && C <= 256 && !(p.variant & 8);
    if ((kLinear || linear4) && tid < 6) smtab[tid] = p.tab[tid / 3][tid % 3];  // visible after the first __syncthreads below

    const int8_t* gsrc = p.grid + env0 * C;
    const uint32_t tile_bytes = (uint32_t)(nG * C);
    const bool bulk_ok = (tile_bytes & 15u) == 0 && ((((uintptr_t)gsrc) & 15u) == 0);
    const bool need_load = !(MODE == MODE_RESET && p.env_mask == nullptr);
    // large grids: a tick changes <= 6 of the C bytes, so only those (or a rebuilt game) go back to HBM
    const bool sparse_wb = C_T == 0 && MODE == MODE_STEP && C >= 2048;  // measured: pays off from ~45x45 up (32x32 is faster written whole)

    if (tid == 0 && bulk_ok && need_load) mbar_init(bar, 1);
    __syncthreads();
    if (need_load) {
        if (bulk_ok) {
            if (tid == 0) { mbar_expect_tx(bar, tile_bytes); bulk_g2s(tile, gsrc, tile_bytes, bar); }
        } else {
            for (uint32_t i = tid; i < tile_bytes; i += NT) tile[i] = gsrc[i];
        }
    }
    // template grid for resets (reference tron/map.py:43-48): border WALL, interior EMPTY
    if (MODE != MODE_OBSERVE) {
        const int Hc = p.Hc, Wc = p.W + 2;
        for (int c = tid; c < C; c += NT) {
            const int r = c / Hc, q = c - r * Hc;
            tmpl[c] = (r == 0 || r == Wc - 1 || q == 0 || q == Hc - 1) ? (int8_t)TRON_TILE_WALL : (int8_t)TRON_TILE_EMPTY;
        }
    }

    const bool owner = tid < nG;
    const long long env = env0 + tid;
    uint2 mraw = make_uint2(0, 0);
    if (owner && MODE != MODE_OBSERVE) mraw = p.meta[env];

    if (need_load && bulk_ok) mbar_wait(bar, 0);
    __syncthreads();

    const int T = MODE == MODE_STEP ? p.T : 1;
    for (int t = 0; t < T; ++t) {
        if (MODE != MODE_OBSERVE) {
            // ------------------------------------------------------------ phase 1: thread-per-game tick
            if (owner) {
                EnvState e = unpack_meta(mraw);
                BoxRegs bx;
                bool do_reset;
                if (C_T == 0 && sparse_wb) {  // large grids: remember the <=6 bytes this tick changes, write only those back
                    LoggedByteCells cells{tile + tid * C, p.Hc, C, 0, {0, 0, 0, 0, 0, 0}, {0, 0, 0, 0, 0, 0}};
                    do_reset = env_tick<MODE, false>(cells, p, e, env, t, tid, bx);
                    if (!do_reset) {
                        int8_t* gg = p.grid + (size_t)env * C;
#pragma unroll
                        for (int k = 0; k < 6; ++k) if (k < cells.n) gg[cells.idx[k]] = cells.val[k];
                    }
                } else {
                    ByteCells cells{tile + tid * C, p.Hc, C};
                    do_reset = env_tick<MODE, false>(cells, p, e, env, t, tid, bx);
                }
                if (MODE == MODE_RESET && do_reset && p.boxes) {  // a fresh grid has exactly two non-template cells
                    box_set_spawn(bx, e);
                    p.boxes[env] = pack_boxes(bx);
                    e.flags |= TRON_FLAG_BOXES_VALID;
                }
                if (do_reset) hidx[tid] = make_ushort2((unsigned short)((e.r1 + 1) * p.Hc + e.c1 + 1), (unsigned short)((e.r2 + 1) * p.Hc + e.c2 + 1));
                mraw = pack_meta(e);
                rflag[tid] = do_reset ? 1 : 0;
            }
            __syncthreads();
            if (LP > 0 && MODE == MODE_STEP && p.obs_term) {  // last frame of the games that just finished, before they are rebuilt
                if constexpr (kLinear) encode_tile_linear144<NT, OD, LP, CP>(tile, nG, env0, p, p.obs_every_tick ? t : 0, smtab, p.obs_term, rflag);
                else if (linear4) encode_tile_linear4<NT, OD, LP, CP>(tile, C, nG, env0, p, p.obs_every_tick ? t : 0, smtab, p.obs_term, rflag);
                else encode_tile<C_T, NT, OD, LP, CP, CH>(tile, nG, env0, p, p.obs_every_tick ? t : 0, p.obs_term, rflag);
                __syncthreads();
            }
            // ------------------------------------------------------------ phase 2: rebuild reset games
            {
                constexpr int V = (C_T != 0 && C_T % 16 == 0) ? 16 : 4;  // template copy granularity (C % 4 == 0 or scalar)
                if ((C % V) == 0) {
                    const int per = C / V;
                    auto fill = [&](int e, int ch) {
                        if (V == 16) ((uint4*)(tile + e * C))[ch] = ((const uint4*)tmpl)[ch];
                        else ((uint32_t*)(tile + e * C))[ch] = ((const uint32_t*)tmpl)[ch];
                        const ushort2 h = hidx[e];
                        if ((int)h.x / V == ch) tile[e * C + h.x] = TRON_TILE_P1_HEAD;
                        if ((int)h.y / V == ch) tile[e * C + h.y] = TRON_TILE_P2_HEAD;
                    };
                    if (C_T == 0 && per >= 4 * NT) {
                        for (int e = 0; e < nG; ++e) {
                            if (!rflag[e]) continue;
                            for (int ch = tid; ch < per; ch += NT) fill(e, ch);
                        }
                    } else {
                        for (int it = tid; it < nG * per; it += NT) {
                            const int e = it / per;
                            if (rflag[e]) fill(e, it - e * per);
                        }
                    }
                } else {
                    for (int it = tid; it < nG * C; it += NT) {
                        const int e = it / C, c = it - e * C;
                        if (!rflag[e]) continue;
                        const ushort2 h = hidx[e];
                        tile[it] = c == h.y ? (int8_t)TRON_TILE_P2_HEAD : c == h.x ? (int8_t)TRON_TILE_P1_HEAD : tmpl[c];
                    }
                }
            }
            if (t == T - 1 && !sparse_wb) fence_proxy_async();
            __syncthreads();
            // ------------------------------------------------------------ write the tile back (last tick only)
            if (sparse_wb) {  // changed bytes already went out in phase 1; rebuilt games are written whole, every tick
                if ((C & 3) == 0) {
                    const int per = C / 4;
                    for (int e = 0; e < nG; ++e) {
                        if (!rflag[e]) continue;
                        uint32_t* gd = (uint32_t*)(p.grid + (size_t)(env0 + e) * C);
                        const uint32_t* sd = (const uint32_t*)(tile + e * C);
                        for (int ch = tid; ch < per; ch += NT) gd[ch] = sd[ch];
                    }
                } else {
                    for (int e = 0; e < nG; ++e) {
                        if (!rflag[e]) continue;
                        for (int ch = tid; ch < C; ch += NT) p.grid[(size_t)(env0 + e) * C + ch] = tile[e * C + ch];
                    }
                }
                if (t == T - 1 && owner) p.meta[env] = mraw;
            } else if (t == T - 1) {
                int8_t* gdst = p.grid + env0 * C;
                if (bulk_ok) {
                    if (tid == 0) { bulk_s2g(gdst, tile, tile_bytes); bulk_commit(); }
                } else {
                    for (uint32_t i = tid; i < tile_bytes; i += NT) gdst[i] = tile[i];
                }
                if (owner) p.meta[env] = mraw;
            }
        }
        // ---------------------------------------------------------------- phase 3: observation planes
        if (MODE == MODE_OBSERVE && owner) emit_extra(p, env);
        if (LP > 0 && (MODE == MODE_OBSERVE || p.obs_every_tick || t == T - 1)) {
            const int tt = (MODE == MODE_STEP && p.obs_every_tick) ? t : 0;
            if constexpr (kLinear) {  // one contiguous 512-byte run per warp store (see step_bits.cu); TRON_OPT_ENCODE_VARIANT 8 = per-plane schedule
                if (!(p.variant & 8)) encode_tile_linear144<NT, OD, LP, CP>(tile, nG, env0, p, tt, smtab);
                else encode_tile<C_T, NT, OD, LP, CP, CH>(tile, nG, env0, p, tt);
            } else if (linear4) {
                encode_tile_linear4<NT, OD, LP, CP>(tile, C, nG, env0, p, tt, smtab);
            } else {
                encode_tile<C_T, NT, OD, LP, CP, CH>(tile, nG, env0, p, tt);
            }
        }
        if (T > 1) __syncthreads();  // next tick's phase 1 rewrites the tile
    }
    if (MODE != MODE_OBSERVE && bulk_ok && !sparse_wb && tid == 0) bulk_wait_read_all();  // tile must outlive the bulk store's read
}

}  // namespace tron
