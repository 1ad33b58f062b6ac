#!/usr/bin/env python
"""How fast does HBM absorb observation rows written only in part?  A standalone nvcc-built kernel writes a buffer the size of the
bench.py headline's observation (4,194,304 games x 576 B: 10x10, bf16, one plane per player) through the same CTA-scan + store loop
as the delta path of step_bits_kernel.

Part 1 (unpadded, 128 games per CTA, 2 x 16-byte streaming stores per unit, as round 3 measured it):
  (a) every 32-byte sector;
  (b) a seeded subset of 32-byte sectors: each of a game's 9 unit positions is dirty with probability 0.351 (the measured mean
      dirty fraction of the headline workload), in both players' planes alike, as the kernel's per-game unit mask is;
  (c) the subset of (b) rounded up to 64-byte pairs.
Part 2 (the matrix): pattern (b) under
  games per CTA G 128 / 256 / 512 / 1024 with 128 or 256 threads (games strided by the thread count, so loads stay coalesced),
  resident CTAs per SM 1-6 and 8, set by padding the dynamic shared memory as smem_for_ctas_per_sm (step_dispatch.cuh) does,
      starting from the shared memory a delta kernel of that G needs (the [G][144] tile, the flags, the tables and the unit list);
      a residency the footprint cannot reach is reported with the residency the occupancy calculator gives and skipped;
  store shape: two lanes x 16 B per unit (st.global.v4) or one lane x 32 B (st.global.v8.b32, STG.E.*.256);
  cache hint: .cs (evict-first) or the default.
Part 3: the three fastest matrix rows and the round-3 configuration (G 128, 128 threads, 5 CTAs per SM, 2 x 16 B, .cs) again,
  with the kernel's coalesced state traffic added: per game 42 B read (planes 32, meta 8, actions 2) and 50 B written (planes 32,
  meta 8, reward 8, done 1, winner 1).  The dirty mask depends on the loaded planes, so the scan waits for the loads as in the kernel.
Part 4: every reachable matrix row with the state traffic.
Prints one JSON line per row (us per pass, useful GB/s = observation bytes actually written / time) with the card, its power limit
and its SM clock, read in the same run.
usage: sector_write_probe.py [--passes 20] [--out FILE.jsonl]"""
import argparse
import json
import os
import subprocess
import tempfile

SRC = r"""
#include <cstdio>
#include <cstdint>
#include <cstdlib>
#include <vector>
#include <algorithm>
#include <cuda_runtime.h>
constexpr int SECT = 18;  // 32-byte sectors per game (576 B)
constexpr long long N = 4194304;
__device__ __host__ __forceinline__ uint32_t mix(uint32_t x) { x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16; return x; }
__device__ __host__ __forceinline__ uint32_t game_mask(long long g, int pattern, uint32_t thr) {
    if (pattern == 0) return (1u << SECT) - 1u;
    uint32_t m = 0;
    for (int u = 0; u < 9; ++u) if (mix((uint32_t)g * 9u + u) < thr) m |= (1u << u) | (1u << (u + 9));
    if (pattern == 2) m |= ((m & 0x15555u) << 1) | ((m & 0x2AAAAu) >> 1);  // round up to 64-byte pairs
    return m;
}
struct State { uint4* planes; uint2* meta; const uchar2* act; float2* reward; int8_t* done; int8_t* winner; };
// G games per CTA, T threads, GPT = G / T games per thread (game = slot * T + tid); V8: one lane per unit with one 32-byte store,
// else two lanes x 16 B; CS: streaming (.cs) stores; ST: plus the coalesced state traffic
template <int G, int T, bool V8, bool CS, bool ST>
__global__ void __launch_bounds__(T) probe(uint4* out, int pattern, uint32_t thr, State s) {
    constexpr int GPT = G / T;
    using Ent = typename std::conditional<(G <= 512), uint16_t, uint32_t>::type;  // game << 5 | unit
    extern __shared__ __align__(16) unsigned char smem[];
    int* wsum = (int*)smem;
    Ent* list = (Ent*)(smem + 64);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long g0 = (long long)blockIdx.x * G;
    uint4 pa[GPT], pb[GPT]; uint2 mt[GPT]; uchar2 ac[GPT];
    if (ST) {
#pragma unroll
        for (int k = 0; k < GPT; ++k) {
            const long long g = g0 + k * T + tid;
            if (g < N) { pa[k] = s.planes[2 * g]; pb[k] = s.planes[2 * g + 1]; mt[k] = s.meta[g]; ac[k] = s.act[g]; }
        }
    }
    int base = 0;
#pragma unroll
    for (int k = 0; k < GPT; ++k) {  // one CTA scan per slot: the list is in game (= address) order
        const long long g = g0 + k * T + tid;
        uint32_t m = g < N ? game_mask(g, pattern, thr) : 0u;
        if (ST && g < N) {
            if (pa[k].x == 0xDEADBEEFu) m = 0u;  // never true (zeroed planes): the mask waits for the loads, as the kernel's does
            s.planes[2 * g] = make_uint4(pa[k].x + 1u, pa[k].y, pa[k].z, pa[k].w ^ ac[k].x);
            s.planes[2 * g + 1] = make_uint4(pb[k].x, pb[k].y + 1u, pb[k].z, pb[k].w ^ ac[k].y);
            s.meta[g] = make_uint2(mt[k].x + 1u, mt[k].y);
            s.reward[g] = make_float2((float)(mt[k].x & 1u), 0.f);
            s.done[g] = (int8_t)(mt[k].y & 1u); s.winner[g] = (int8_t)(ac[k].x & 1u);
        }
        const int c = __popc(m);
        int incl = c;
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += v; }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        int off = base + incl - c, total = 0;
        for (int w = 0; w < T / 32; ++w) { off += w < warp ? wsum[w] : 0; total += wsum[w]; }
        for (uint32_t q = m; q; q &= q - 1u) list[off++] = (Ent)(((k * T + tid) << 5) | (__ffs(q) - 1));
        base += total;
        __syncthreads();
    }
    const int total = base;
    if (V8) {
        for (int i = tid; i < total; i += T) {
            const uint32_t e = list[i];
            const unsigned long long a = (unsigned long long)(out + (g0 + (e >> 5)) * (2 * SECT) + (e & 31u) * 2);
            if (CS) asm volatile("st.global.cs.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" :: "l"(a), "r"(i), "r"(e), "r"(0), "r"(0), "r"(i), "r"(e), "r"(0), "r"(0) : "memory");
            else asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" :: "l"(a), "r"(i), "r"(e), "r"(0), "r"(0), "r"(i), "r"(e), "r"(0), "r"(0) : "memory");
        }
    } else {
        for (int i = tid; i < 2 * total; i += T) {
            const uint32_t e = list[i >> 1];
            uint4* a = out + (g0 + (e >> 5)) * (2 * SECT) + (e & 31u) * 2 + (i & 1);
            const uint4 v = make_uint4((uint32_t)i, e, 0u, 0u);
            if (CS) __stcs(a, v); else *a = v;
        }
    }
}
// shared memory of a delta kernel with G games per CTA: [G][144] tile, [G] flags, 6 tables, warp sums, [G * 18] unit list
static size_t kernel_smem(int G) { return (size_t)G * 144 + ((G + 15) & ~15) + 96 + 64 + (size_t)G * SECT * (G <= 512 ? 2 : 4); }
static size_t smem_for_ctas_per_sm(size_t smem, long long cap) {  // step_dispatch.cuh
    const size_t want = (size_t)(228 * 1024) / (size_t)(cap + 1) - 1024 + 256;
    return want > smem && want <= 200 * 1024 ? want : smem;
}
struct Row { const char* pattern; int G, T, cap, resident; size_t smem; bool v8, cs, st; double us; long long sect; };
static uint4* g_buf; static State g_st; static uint32_t g_thr; static int g_passes;
static long long g_sect[3];
template <int G, int T, bool V8, bool CS, bool ST>
static bool run(int pattern, int cap, bool pad, Row& r) {
    auto k = probe<G, T, V8, CS, ST>;
    // unpadded: only the unit list, as round 3 ran it
    const size_t smem = pad ? smem_for_ctas_per_sm(kernel_smem(G), cap) : 64 + (size_t)G * SECT * (G <= 512 ? 2 : 4);
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int res = 0; cudaOccupancyMaxActiveBlocksPerMultiprocessor(&res, k, T, smem);
    r = Row{pattern == 0 ? "a: every 32-byte sector" : pattern == 1 ? "b: seeded 32-byte sectors" : "c: (b) rounded up to 64-byte pairs",
            G, T, cap, res, smem, V8, CS, ST, 0.0, g_sect[pattern]};
    if (pad && res != cap) return false;
    const unsigned grid = (unsigned)((N + G - 1) / G);
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    for (int w = 0; w < 3; ++w) k<<<grid, T, smem>>>(g_buf, pattern, g_thr, g_st);
    cudaEventRecord(a);
    for (int p = 0; p < g_passes; ++p) k<<<grid, T, smem>>>(g_buf, pattern, g_thr, g_st);
    cudaEventRecord(b); cudaEventSynchronize(b);
    float ms = 0; cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a); cudaEventDestroy(b);
    r.us = 1e3 * ms / g_passes;
    return true;
}
static void print(const Row& r, const char* part) {
    const double wbytes = (double)r.sect * 32.0, bytes = (double)N * SECT * 32;
    printf("{\"part\": \"%s\", \"pattern\": \"%s\", \"games_per_cta\": %d, \"threads\": %d, \"ctas_per_sm\": %d, \"resident_ctas_per_sm\": %d, "
           "\"smem\": %zu, \"store\": \"%s\", \"hint\": \"%s\", \"state\": %s, \"buffer_bytes\": %.0f, \"written_bytes\": %.0f, "
           "\"written_fraction\": %.4f, \"us_per_pass\": %.1f, \"useful_GBps\": %.1f, \"passes\": %d, \"cuda_error\": \"%s\"}\n",
           part, r.pattern, r.G, r.T, r.cap, r.resident, r.smem, r.v8 ? "1x32B" : "2x16B", r.cs ? "cs" : "default", r.st ? "true" : "false",
           bytes, wbytes, wbytes / bytes, r.us, r.us > 0 ? wbytes / (r.us * 1e3) : 0.0, g_passes, cudaGetErrorString(cudaGetLastError()));
    fflush(stdout);
}
// one configuration key -> the template instantiation
template <bool ST>
static bool dispatch(int G, int T, bool v8, bool cs, int pattern, int cap, bool pad, Row& r) {
#define P_CASE(g, t) if (G == g && T == t) { \
        if (v8) return cs ? run<g, t, true, true, ST>(pattern, cap, pad, r) : run<g, t, true, false, ST>(pattern, cap, pad, r); \
        return cs ? run<g, t, false, true, ST>(pattern, cap, pad, r) : run<g, t, false, false, ST>(pattern, cap, pad, r); }
    P_CASE(128, 128) P_CASE(256, 128) P_CASE(256, 256) P_CASE(512, 128) P_CASE(512, 256) P_CASE(1024, 128) P_CASE(1024, 256)
#undef P_CASE
    return false;
}
int main(int argc, char** argv) {
    g_passes = atoi(argv[1]);
    g_thr = (uint32_t)(0.351 * 4294967296.0);
    const size_t bytes = (size_t)N * SECT * 32;
    if (cudaMalloc(&g_buf, bytes) != cudaSuccess) { printf("{\"error\": \"cudaMalloc\"}\n"); return 1; }
    cudaMemset(g_buf, 0, bytes);
    cudaMalloc(&g_st.planes, N * 32); cudaMemset(g_st.planes, 0, N * 32);
    cudaMalloc(&g_st.meta, N * 8); cudaMemset(g_st.meta, 0, N * 8);
    uchar2* act; cudaMalloc(&act, N * 2); cudaMemset(act, 0, N * 2); g_st.act = act;
    cudaMalloc(&g_st.reward, N * 8); cudaMalloc(&g_st.done, N); cudaMalloc(&g_st.winner, N);
    for (int pat = 0; pat < 3; ++pat) {  // sectors written per pass, counted on the host with the same hash
        long long s = 0;
        for (long long g = 0; g < N; ++g) s += __builtin_popcount(game_mask(g, pat, g_thr));
        g_sect[pat] = s;
    }
    Row r;
    for (int pat = 0; pat < 3; ++pat) { run<128, 128, false, true, false>(pat, 0, false, r); r.cap = 0; print(r, "1: round 3, unpadded"); }
    std::vector<Row> rows;
    const int Gs[4] = {128, 256, 512, 1024}, caps[7] = {1, 2, 3, 4, 5, 6, 8};
    for (int G : Gs) for (int T : {128, 256}) {
        if (T > G) continue;
        for (int cap : caps) for (int v8 = 0; v8 < 2; ++v8) for (int cs = 1; cs >= 0; --cs) {
            if (dispatch<false>(G, T, v8, cs, 1, cap, true, r)) { print(r, "2: matrix"); rows.push_back(r); }
            else print(r, "2: matrix, residency not reachable");
        }
    }
    std::sort(rows.begin(), rows.end(), [](const Row& x, const Row& y) { return x.us < y.us; });
    std::vector<Row> pick(rows.begin(), rows.begin() + std::min<size_t>(3, rows.size()));
    pick.push_back(Row{"", 128, 128, 5, 0, 0, false, true, false, 0, 0});
    for (const Row& q : pick) {  // each twice in a row, the state-free twin first, so that both read the same moment of the card
        print(r, dispatch<false>(q.G, q.T, q.v8, q.cs, 1, q.cap, true, r) ? "3: pattern (b) alone" : "3: residency not reachable");
        print(r, dispatch<true>(q.G, q.T, q.v8, q.cs, 1, q.cap, true, r) ? "3: pattern (b) + state" : "3: residency not reachable");
    }
    for (const Row& q : rows)  // the whole matrix with the state traffic: the best write-only rows need not be the best with it
        if (dispatch<true>(q.G, q.T, q.v8, q.cs, 1, q.cap, true, r)) print(r, "4: matrix + state");
        else print(r, "4: matrix + state, residency not reachable");
    return 0;
}
"""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    smi = ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"]
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "probe.cu"), os.path.join(d, "probe")
        with open(src, "w") as f:
            f.write(SRC)
        subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe, src], check=True)
        card = subprocess.run(smi, capture_output=True, text=True).stdout.strip()
        res = subprocess.run([exe, str(a.passes)], capture_output=True, text=True, check=True).stdout
        card_after = subprocess.run(smi, capture_output=True, text=True).stdout.strip()
    meta = {"card": card, "card_after": card_after, "query": q}
    lines = [json.dumps(dict(json.loads(l), **meta)) for l in res.splitlines() if l.strip()]
    print("\n".join(lines))
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
