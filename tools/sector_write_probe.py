#!/usr/bin/env python
"""How fast does HBM absorb observation rows written only in part?  A standalone nvcc-built kernel writes a buffer the size of the
bench.py headline's observation (4,194,304 games x 576 B: 10x10, bf16, one plane per player) in three patterns, each through the
same CTA-scan + 16-byte streaming-store loop as the delta path of step_bits_kernel:
  (a) every 32-byte sector;
  (b) a seeded subset of 32-byte sectors: each of a game's 9 unit positions is dirty with probability 0.351 (the measured mean
      dirty fraction of the headline workload), in both players' planes alike, as the kernel's per-game unit mask is;
  (c) the subset of (b) rounded up to 64-byte pairs.
Prints one JSON line per pattern (useful GB/s = bytes actually written / time, us per pass) with the card and its power limit.
usage: sector_write_probe.py [--passes 20] [--out FILE.jsonl]"""
import argparse
import json
import os
import subprocess
import tempfile

SRC = r"""
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
constexpr int G = 128, SECT = 18;  // games per CTA, 32-byte sectors per game (576 B)
__device__ __forceinline__ uint32_t mix(uint32_t x) { x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16; return x; }
__global__ void __launch_bounds__(G) probe(uint4* out, long long n, int pattern, uint32_t thr) {
    __shared__ int wsum[G / 32];
    __shared__ uint16_t list[G * SECT];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long g0 = (long long)blockIdx.x * G;
    uint32_t m = 0;
    if (g0 + tid < n) {
        if (pattern == 0) m = (1u << SECT) - 1u;
        else {
            for (int u = 0; u < 9; ++u) if (mix((uint32_t)(g0 + tid) * 9u + u) < thr) m |= (1u << u) | (1u << (u + 9));
            if (pattern == 2) m |= ((m & 0x15555u) << 1) | ((m & 0x2AAAAu) >> 1);  // round up to 64-byte pairs
        }
    }
    const int c = __popc(m);
    int incl = c;
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    int off = incl - c, total = 0;
    for (int w = 0; w < G / 32; ++w) { off += w < warp ? wsum[w] : 0; total += wsum[w]; }
    for (uint32_t k = m; k; k &= k - 1u) list[off++] = (uint16_t)((tid << 5) | (__ffs(k) - 1));
    __syncthreads();
    for (int i = tid; i < 2 * total; i += G) {
        const uint32_t e = list[i >> 1];
        const long long chunk = (g0 + (e >> 5)) * (2 * SECT) + (e & 31u) * 2 + (i & 1);
        __stcs(out + chunk, make_uint4((uint32_t)i, e, 0u, 0u));
    }
}
int main(int argc, char** argv) {
    const long long n = 4194304; const int passes = atoi(argv[1]);
    const uint32_t thr = (uint32_t)(0.351 * 4294967296.0);
    uint4* buf; size_t bytes = (size_t)n * SECT * 32;
    if (cudaMalloc(&buf, bytes) != cudaSuccess) { printf("{\"error\": \"cudaMalloc\"}\n"); return 1; }
    cudaMemset(buf, 0, bytes);
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    const unsigned grid = (unsigned)((n + G - 1) / G);
    const char* names[3] = {"a: every 32-byte sector", "b: seeded 32-byte sectors", "c: (b) rounded up to 64-byte pairs"};
    for (int pat = 0; pat < 3; ++pat) {
        long long sect = 0;  // sectors written per pass, counted on the host with the same hash
        for (long long g = 0; g < n; ++g) {
            uint32_t m = 0;
            if (pat == 0) m = (1u << SECT) - 1u;
            else {
                for (int u = 0; u < 9; ++u) {
                    uint32_t x = (uint32_t)g * 9u + u; x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
                    if (x < thr) m |= (1u << u) | (1u << (u + 9));
                }
                if (pat == 2) m |= ((m & 0x15555u) << 1) | ((m & 0x2AAAAu) >> 1);
            }
            sect += __builtin_popcount(m);
        }
        for (int w = 0; w < 3; ++w) probe<<<grid, G>>>(buf, n, pat, thr);
        cudaEventRecord(a);
        for (int p = 0; p < passes; ++p) probe<<<grid, G>>>(buf, n, pat, thr);
        cudaEventRecord(b); cudaEventSynchronize(b);
        float ms = 0; cudaEventElapsedTime(&ms, a, b);
        const double us = 1e3 * ms / passes, wbytes = (double)sect * 32.0;
        printf("{\"pattern\": \"%s\", \"buffer_bytes\": %zu, \"written_bytes\": %.0f, \"written_fraction\": %.4f, \"us_per_pass\": %.1f, "
               "\"useful_GBps\": %.1f, \"passes\": %d, \"cuda_error\": \"%s\"}\n",
               names[pat], bytes, wbytes, wbytes / (double)bytes, us, wbytes / (us * 1e3), passes, cudaGetErrorString(cudaGetLastError()));
    }
    cudaFree(buf);
    return 0;
}
"""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "probe.cu"), os.path.join(d, "probe")
        with open(src, "w") as f:
            f.write(SRC)
        subprocess.run([nvcc, "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe, src], check=True)
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True).stdout.strip()
        res = subprocess.run([exe, str(a.passes)], capture_output=True, text=True, check=True).stdout
    lines = [json.dumps(dict(json.loads(l), card=q)) for l in res.splitlines() if l.strip()]
    print("\n".join(lines))
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
