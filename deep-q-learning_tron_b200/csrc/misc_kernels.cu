// misc_kernels.cu -- export/import of env state, action policies, replay ring push/gather/sample.
#include <cuda_bf16.h>

#include "common.cuh"
#include "launch.h"

namespace tron {

// ------------------------------------------------------------------------------------------------
// state export / import (history, drop-in shims, tests)
// ------------------------------------------------------------------------------------------------
__global__ void export_meta_kernel(const uint2* __restrict__ meta, int n, int8_t* heads, uint8_t* alive, uint8_t* done,
                                   uint8_t* winner, int32_t* ep_len) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const uint2 m = meta[e];
    const uint32_t f = m.y & 0xFFu;
    if (heads) ((uint32_t*)heads)[e] = m.x;
    if (alive) { alive[2 * e] = f & 1u; alive[2 * e + 1] = (f >> 1) & 1u; }
    if (done) done[e] = (f >> 2) & 1u;
    if (winner) winner[e] = (f >> TRON_FLAG_WINNER_SHIFT) & 3u;
    if (ep_len) ep_len[e] = (int32_t)(m.y >> 16);
}

__global__ void import_meta_kernel(uint2* __restrict__ meta, int n, int W, int H, const int8_t* heads, const uint8_t* alive,
                                   const uint8_t* done, const uint8_t* winner, const int32_t* ep_len, const int8_t* tiles_for_heads) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    uint2 m = meta[e];
    uint32_t f = m.y & 0xFFu;
    uint32_t k = m.y >> 16;
    if (heads) {  // clamp to the representable range [-1, W] x [-1, H]: a head outside it would index outside the game's cells
        const int8_t* h = heads + 4 * (size_t)e;
        const int r1 = min(max((int)h[0], -1), W), c1 = min(max((int)h[1], -1), H), r2 = min(max((int)h[2], -1), W), c2 = min(max((int)h[3], -1), H);
        m.x = (uint32_t)(uint8_t)r1 | ((uint32_t)(uint8_t)c1 << 8) | ((uint32_t)(uint8_t)r2 << 16) | ((uint32_t)(uint8_t)c2 << 24);
    }
    else if (tiles_for_heads) {  // a grid given without a head array: the heads are where its head tiles are
        uint32_t packed;
        if (heads_from_tiles(tiles_for_heads + (size_t)e * (W + 2) * (H + 2), W, H, packed)) m.x = packed;
    }
    if (alive) f = (f & ~3u) | (alive[2 * e] ? 1u : 0u) | (alive[2 * e + 1] ? 2u : 0u);
    if (done) f = (f & ~TRON_FLAG_DONE) | (done[e] ? TRON_FLAG_DONE : 0u);
    if (winner) f = (f & ~(3u << TRON_FLAG_WINNER_SHIFT)) | ((winner[e] & 3u) << TRON_FLAG_WINNER_SHIFT);
    if (ep_len) k = (uint32_t)ep_len[e] & 0xFFFFu;
    f &= ~0x20u;  // TRON_FLAG_BOXES_VALID: an imported grid has unknown dirty boxes
    m.y = f | (k << 16);
    meta[e] = m;
}

int launch_export_meta(const void* meta, int n, int8_t* heads, uint8_t* alive, uint8_t* done, uint8_t* winner,
                       int32_t* ep_len, cudaStream_t s) {
    export_meta_kernel<<<(n + 255) / 256, 256, 0, s>>>((const uint2*)meta, n, heads, alive, done, winner, ep_len);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}
int launch_import_meta(void* meta, int n, int W, int H, const int8_t* heads, const uint8_t* alive, const uint8_t* done,
                       const uint8_t* winner, const int32_t* ep_len, const int8_t* tiles_for_heads, cudaStream_t s) {
    import_meta_kernel<<<(n + 255) / 256, 256, 0, s>>>((uint2*)meta, n, W, H, heads, alive, done, winner, ep_len, tiles_for_heads);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

// ------------------------------------------------------------------------------------------------
// policies
// ------------------------------------------------------------------------------------------------
__global__ void advance_counter_kernel(unsigned long long* c, unsigned long long delta) { *c += delta; }
int launch_advance_counter(uint64_t* c, uint64_t delta, cudaStream_t s) {
    advance_counter_kernel<<<1, 1, 0, s>>>((unsigned long long*)c, delta);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

__global__ void random_actions_kernel(uint8_t* actions, int n, unsigned long long seed, unsigned long long counter,
                                      const unsigned long long* counter_dev, unsigned long long base) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    if (counter_dev) counter += *counter_dev;
    const uint4 r = philox(seed, counter, base + (unsigned long long)e, TAG_ACTION, 0);
    ((uchar2*)actions)[e] = make_uchar2((unsigned char)(r.x >> 30), (unsigned char)(r.y >> 30));
}

// epsilon-greedy (reference DDQN.py:90-110): explore iff u <= eps, else first argmax of the 4 q-values
template <typename QT>
__global__ void select_actions_kernel(const QT* __restrict__ q, int n, float eps, uint8_t* actions, unsigned long long seed,
                                      unsigned long long counter, const unsigned long long* counter_dev, unsigned long long base) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (counter_dev) counter += *counter_dev;
    float v[4];
    if constexpr (sizeof(QT) == 4) {
        const float4 f = ((const float4*)q)[i];
        v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
    } else {
        const uint2 w = ((const uint2*)q)[i];
        v[0] = __uint_as_float(w.x << 16); v[1] = __uint_as_float(w.x & 0xFFFF0000u);
        v[2] = __uint_as_float(w.y << 16); v[3] = __uint_as_float(w.y & 0xFFFF0000u);
    }
    const uint4 r = philox(seed, counter, base + (unsigned long long)i, TAG_EPS, 0);
    const float u = (float)(r.x >> 8) * (1.0f / 16777216.0f);
    int best = 0;
#pragma unroll
    for (int j = 1; j < 4; ++j) if (v[j] > v[best]) best = j;
    actions[i] = (uint8_t)(u <= eps ? (r.y >> 30) : (uint32_t)best);
}

int launch_random_actions(uint8_t* actions, int n, uint64_t seed, uint64_t counter, const uint64_t* cdev, uint64_t base, cudaStream_t s) {
    random_actions_kernel<<<(n + 255) / 256, 256, 0, s>>>(actions, n, seed, counter, (const unsigned long long*)cdev, base);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}
int launch_select_actions(const void* q, int q_dtype, int n, float eps, uint8_t* actions, uint64_t seed, uint64_t counter,
                          const uint64_t* cdev, uint64_t base, cudaStream_t s) {
    const unsigned long long* cd = (const unsigned long long*)cdev;
    if (q_dtype == TRON_F32) select_actions_kernel<float><<<(n + 255) / 256, 256, 0, s>>>((const float*)q, n, eps, actions, seed, counter, cd, base);
    else if (q_dtype == TRON_BF16) select_actions_kernel<uint16_t><<<(n + 255) / 256, 256, 0, s>>>((const uint16_t*)q, n, eps, actions, seed, counter, cd, base);
    else return TRON_ERR_INVALID;
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

// pop_up (reference tron/util.py:11-37) on already-encoded observations: [n, cells] -> [n, 3, cells] planes
// wall = (o == -1); my = 1 if o == -2, 10 if o == 10; enemy = 1 if o == -3, 10 if o == -10.
__global__ void pop_up_kernel(const void* __restrict__ obs, int in_dtype, long long n_maps, int cells, void* planes, int out_dtype) {
    const long long total = n_maps * cells;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        float o;
        if (in_dtype == TRON_F32) o = ((const float*)obs)[i];
        else if (in_dtype == TRON_BF16) o = __uint_as_float((uint32_t)((const uint16_t*)obs)[i] << 16);
        else if (in_dtype == TRON_I8) o = (float)((const int8_t*)obs)[i];
        else if (in_dtype == TRON_I32) o = (float)((const int32_t*)obs)[i];
        else o = (float)((const long long*)obs)[i];
        const float w = o == -1.f ? 1.f : 0.f;
        const float m = o == -2.f ? 1.f : o == 10.f ? 10.f : 0.f;
        const float e = o == -3.f ? 1.f : o == -10.f ? 10.f : 0.f;
        const long long map = i / cells, c = i - map * cells;
        const long long b = map * 3 * cells + c;
        if (out_dtype == TRON_F32) { ((float*)planes)[b] = w; ((float*)planes)[b + cells] = m; ((float*)planes)[b + 2 * cells] = e; }
        else if (out_dtype == TRON_BF16) {
            ((__nv_bfloat16*)planes)[b] = __float2bfloat16_rn(w); ((__nv_bfloat16*)planes)[b + cells] = __float2bfloat16_rn(m);
            ((__nv_bfloat16*)planes)[b + 2 * cells] = __float2bfloat16_rn(e);
        } else { ((int8_t*)planes)[b] = (int8_t)w; ((int8_t*)planes)[b + cells] = (int8_t)m; ((int8_t*)planes)[b + 2 * cells] = (int8_t)e; }
    }
}
int launch_pop_up(const void* obs, int in_dtype, int64_t n_maps, int cells, void* planes, int out_dtype, cudaStream_t s) {
    const long long total = n_maps * cells;
    const int blocks = (int)min((long long)sm_count() * 16, (total + 255) / 256);
    pop_up_kernel<<<blocks, 256, 0, s>>>(obs, in_dtype, n_maps, cells, planes, out_dtype);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

// ------------------------------------------------------------------------------------------------
// replay ring.  A batched step yields 2N transitions whose frames are already contiguous
// ([N,2,P,C] == [2N, frame]), so push is a wrapped streaming copy and gather a row gather.
// ------------------------------------------------------------------------------------------------
// copy n frames of `fb` bytes (fb % 16 == 0) into ring slots (cursor+i) % capacity; one warp per frame chunk
__global__ void replay_push_frames_kernel(uint4* __restrict__ ring_s, uint4* __restrict__ ring_s2, const uint4* __restrict__ s,
                                          const uint4* __restrict__ s2, long long n, int vec_per_frame,
                                          unsigned long long cursor, long long capacity) {
    const long long total = n * vec_per_frame;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long f = i / vec_per_frame;
        const int v = (int)(i - f * vec_per_frame);
        const long long slot = (long long)((cursor + (unsigned long long)f) % (unsigned long long)capacity);
        if (!TRON_DCHECK(slot >= 0 && slot < capacity, DBG_RING_SLOT)) continue;
        const uint4 a = __ldcs(s + i), b = __ldcs(s2 + i);
        ring_s[slot * vec_per_frame + v] = a;
        ring_s2[slot * vec_per_frame + v] = b;
    }
}
__global__ void replay_push_frames_bytes_kernel(uint8_t* ring_s, uint8_t* ring_s2, const uint8_t* s, const uint8_t* s2, long long n,
                                                long long fb, unsigned long long cursor, long long capacity) {
    const long long total = n * fb;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long f = i / fb, v = i - f * fb;
        const long long slot = (long long)((cursor + (unsigned long long)f) % (unsigned long long)capacity);
        ring_s[slot * fb + v] = s[i];
        ring_s2[slot * fb + v] = s2[i];
    }
}
__global__ void replay_push_scalars_kernel(uint8_t* ring_a, float* ring_r, uint8_t* ring_d, const uint8_t* a, const float* r,
                                           const uint8_t* d, int done_stride, long long n, unsigned long long cursor,
                                           long long capacity) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long slot = (long long)((cursor + (unsigned long long)i) % (unsigned long long)capacity);
    ring_a[slot] = a[i];
    ring_r[slot] = r[i];
    ring_d[slot] = d[done_stride == 2 ? i / 2 : i];
}

int launch_replay_push(const replay_ring* ring, uint64_t cursor, const void* s, const void* s2, const uint8_t* action,
                       const float* reward, const uint8_t* done, int done_stride, int64_t n, cudaStream_t st) {
    const long long es = tron_dtype_size(ring->frame_dtype);
    const long long fb = (long long)ring->frame_elems * es;
    const bool vec = (fb % 16 == 0) && ((((uintptr_t)s | (uintptr_t)s2 | (uintptr_t)ring->state | (uintptr_t)ring->next_state) & 15u) == 0);
    if (vec) {
        const long long total = n * (fb / 16);
        const int blocks = (int)min((long long)sm_count() * 16, (total + 255) / 256);
        replay_push_frames_kernel<<<blocks, 256, 0, st>>>((uint4*)ring->state, (uint4*)ring->next_state, (const uint4*)s, (const uint4*)s2, n,
                                                          (int)(fb / 16), cursor, ring->capacity);
    } else {
        const long long total = n * fb;
        const int blocks = (int)min((long long)sm_count() * 16, (total + 255) / 256);
        replay_push_frames_bytes_kernel<<<blocks, 256, 0, st>>>((uint8_t*)ring->state, (uint8_t*)ring->next_state, (const uint8_t*)s,
                                                                (const uint8_t*)s2, n, fb, cursor, ring->capacity);
    }
    replay_push_scalars_kernel<<<(int)((n + 255) / 256), 256, 0, st>>>(ring->action, ring->reward, ring->done, action, reward, done,
                                                                      done_stride, n, cursor, ring->capacity);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

// uniform sampling without replacement: feistel_make / feistel_apply (common.cuh)
__global__ void replay_sample_kernel(long long size, long long k, unsigned long long seed, unsigned long long counter, long long* idx) {
    const FeistelPerm f = feistel_make((unsigned long long)size, seed, counter);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < k; i += (long long)gridDim.x * blockDim.x)
        idx[i] = (long long)feistel_apply(f, (unsigned long long)i);
}
int launch_replay_sample(int64_t size, int64_t k, uint64_t seed, uint64_t counter, int64_t* idx, cudaStream_t st) {
    const int blocks = (int)min((long long)sm_count() * 8, (long long)((k + 127) / 128));
    replay_sample_kernel<<<blocks, 128, 0, st>>>(size, k, seed, counter, (long long*)idx);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

// ------------------------------------------------------------------------------------------------
// gather: one CTA per sampled transition; converts frame dtype -> out dtype (f32 | bf16)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float load_f32(const void* p, int dt, long long i) {
    if (dt == TRON_F32) return ((const float*)p)[i];
    if (dt == TRON_BF16) return __uint_as_float((uint32_t)((const uint16_t*)p)[i] << 16);
    return (float)((const int8_t*)p)[i];
}
__device__ __forceinline__ void store_out(void* p, int dt, long long i, float v) {
    if (dt == TRON_F32) ((float*)p)[i] = v;
    else ((__nv_bfloat16*)p)[i] = __float2bfloat16_rn(v);
}
// copy/convert the two frames of one transition: src_s / src_s2 point at the frames (F elements of dtype fd), row = output row
__device__ __forceinline__ void gather_frames(const void* src_s, const void* src_s2, int fd, int F, void* out_s, void* out_s2, int out_dtype, long long row) {
    const bool al = ((((uintptr_t)src_s | (uintptr_t)src_s2) & 15u) == 0);
    if (fd == out_dtype && ((size_t)F * tron_elem(fd)) % 16 == 0 && al) {  // same dtype: 16-byte row copy
        const int nv = (int)((size_t)F * tron_elem(fd) / 16);
        const uint4* a = (const uint4*)src_s;
        const uint4* b = (const uint4*)src_s2;
        uint4* oa = (uint4*)((char*)out_s + (size_t)row * F * tron_elem(fd));
        uint4* ob = (uint4*)((char*)out_s2 + (size_t)row * F * tron_elem(fd));
        for (int v = threadIdx.x; v < nv; v += blockDim.x) { oa[v] = a[v]; ob[v] = b[v]; }
    } else if (fd == TRON_BF16 && out_dtype == TRON_F32 && F % 8 == 0 && al) {  // bf16 ring -> f32 batch: 16-byte loads, 2 x 16-byte stores
        const int nv = F / 8;
        const uint4* a = (const uint4*)src_s;
        const uint4* b = (const uint4*)src_s2;
        uint4* oa = (uint4*)((float*)out_s + (size_t)row * F);
        uint4* ob = (uint4*)((float*)out_s2 + (size_t)row * F);
        for (int v = threadIdx.x; v < nv; v += blockDim.x) {
            const uint4 x = a[v], y = b[v];
            oa[2 * v] = make_uint4(x.x << 16, x.x & 0xFFFF0000u, x.y << 16, x.y & 0xFFFF0000u);
            oa[2 * v + 1] = make_uint4(x.z << 16, x.z & 0xFFFF0000u, x.w << 16, x.w & 0xFFFF0000u);
            ob[2 * v] = make_uint4(y.x << 16, y.x & 0xFFFF0000u, y.y << 16, y.y & 0xFFFF0000u);
            ob[2 * v + 1] = make_uint4(y.z << 16, y.z & 0xFFFF0000u, y.w << 16, y.w & 0xFFFF0000u);
        }
    } else {
        for (int j = threadIdx.x; j < F; j += blockDim.x) {
            store_out(out_s, out_dtype, row * F + j, load_f32(src_s, fd, j));
            store_out(out_s2, out_dtype, row * F + j, load_f32(src_s2, fd, j));
        }
    }
}
__device__ __forceinline__ void gather_ring_row(const replay_ring& ring, long long slot, long long row, void* out_s, void* out_s2, int out_dtype,
                                                long long* out_a, float* out_r, float* out_d) {
    if (!TRON_DCHECK(slot >= 0 && slot < (long long)ring.capacity, DBG_RING_SLOT)) return;
    const size_t fb = (size_t)ring.frame_elems * tron_elem(ring.frame_dtype);
    gather_frames((const char*)ring.state + (size_t)slot * fb, (const char*)ring.next_state + (size_t)slot * fb, ring.frame_dtype, ring.frame_elems,
                  out_s, out_s2, out_dtype, row);
    if (threadIdx.x == 0) {
        out_a[row] = (long long)ring.action[slot];
        out_r[row] = ring.reward[slot];
        out_d[row] = (float)ring.done[slot];
    }
}
__global__ void replay_gather_kernel(const replay_ring ring, const long long* __restrict__ idx, long long k, void* out_s, void* out_s2,
                                     int out_dtype, long long* out_a, float* out_r, float* out_d) {
    const long long row = blockIdx.x;
    if (row >= k) return;
    const long long slot = min(max(idx[row], 0ll), (long long)ring.capacity - 1);  // a bad index must not read outside the ring
    gather_ring_row(ring, slot, row, out_s, out_s2, out_dtype, out_a, out_r, out_d);
}
int launch_replay_gather(const replay_ring* ring, const int64_t* idx, int64_t k, void* out_s, void* out_s2, int out_dtype,
                         int64_t* out_a, float* out_r, float* out_d, cudaStream_t st) {
    replay_gather_kernel<<<(unsigned)k, 128, 0, st>>>(*ring, (const long long*)idx, k, out_s, out_s2, out_dtype, (long long*)out_a, out_r, out_d);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

// sampling fused into the gather: CTA `row` evaluates pi(row) itself (ReplayBuffer.sample, DDQN.py:191-200, in one launch)
__global__ void replay_sample_gather_kernel(const replay_ring ring, long long size, long long k, unsigned long long seed, unsigned long long counter,
                                            void* out_s, void* out_s2, int out_dtype, long long* out_a, float* out_r, float* out_d, long long* out_idx) {
    const long long row = blockIdx.x;
    if (row >= k) return;
    const long long slot = (long long)feistel_apply(feistel_make((unsigned long long)size, seed, counter), (unsigned long long)row);
    if (out_idx && threadIdx.x == 0) out_idx[row] = slot;
    gather_ring_row(ring, slot, row, out_s, out_s2, out_dtype, out_a, out_r, out_d);
}
int launch_replay_sample_gather(const replay_ring* ring, int64_t size, int64_t k, uint64_t seed, uint64_t counter, void* out_s, void* out_s2,
                                int out_dtype, int64_t* out_a, float* out_r, float* out_d, int64_t* out_idx, cudaStream_t st) {
    replay_sample_gather_kernel<<<(unsigned)k, 128, 0, st>>>(*ring, size, k, seed, counter, out_s, out_s2, out_dtype, (long long*)out_a, out_r, out_d,
                                                            (long long*)out_idx);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

// frame-sharing ring: transition (tick, row) from window_transition (common.cuh); state = frames[tick % S][row], next_state =
// terminal[tick % S][row] if the env finished at that tick (and terminal frames are kept) else frames[(tick+1) % S][row]
__global__ void replay_frames_sample_gather_kernel(const replay_frames fr, long long first_tick, long long n_ticks, long long k, unsigned long long seed,
                                                   unsigned long long counter, void* out_s, void* out_s2, int out_dtype, long long* out_a, float* out_r,
                                                   float* out_d, long long* out_idx) {
    const long long row = blockIdx.x;
    if (row >= k) return;
    const longlong2 tr = window_transition(first_tick, n_ticks, fr.rows, seed, counter, row);
    const long long tick = tr.x, r = tr.y;
    const long long slot = tick % fr.n_slots, nslot = (tick + 1) % fr.n_slots;
    if (!TRON_DCHECK(slot >= 0 && slot < fr.n_slots && r >= 0 && r < fr.rows, DBG_RING_SLOT)) return;
    const size_t fb = (size_t)fr.frame_elems * tron_elem(fr.frame_dtype);
    const uint8_t dn = fr.done[slot * (fr.rows / 2) + r / 2];
    const char* s1 = (const char*)fr.frames + ((size_t)slot * fr.rows + r) * fb;
    const char* s2 = (dn && fr.terminal) ? (const char*)fr.terminal + ((size_t)slot * fr.rows + r) * fb : (const char*)fr.frames + ((size_t)nslot * fr.rows + r) * fb;
    gather_frames(s1, s2, fr.frame_dtype, fr.frame_elems, out_s, out_s2, out_dtype, row);
    if (threadIdx.x == 0) {
        out_a[row] = (long long)fr.action[slot * fr.rows + r];
        out_r[row] = fr.reward[slot * fr.rows + r];
        out_d[row] = (float)dn;
        if (out_idx) out_idx[row] = tick * fr.rows + r;
    }
}
int launch_replay_frames_sample_gather(const replay_frames* fr, int64_t first_tick, int64_t n_ticks, int64_t k, uint64_t seed, uint64_t counter,
                                       void* out_s, void* out_s2, int out_dtype, int64_t* out_a, float* out_r, float* out_d, int64_t* out_idx,
                                       cudaStream_t st) {
    replay_frames_sample_gather_kernel<<<(unsigned)k, 128, 0, st>>>(*fr, first_tick, n_ticks, k, seed, counter, out_s, out_s2, out_dtype, (long long*)out_a,
                                                                   out_r, out_d, (long long*)out_idx);
    return cudaGetLastError() == cudaSuccess ? TRON_OK : TRON_ERR_CUDA;
}

// ------------------------------------------------------------------------------------------------
// debug-build violation counters (see common.cuh)
// ------------------------------------------------------------------------------------------------
#ifdef TRON_DEBUG
typedef int (*dbg_reader)(unsigned long long*, int*);
static dbg_reader* dbg_readers(int** n) {
    static dbg_reader r[32];
    static int count = 0;
    *n = &count;
    return r;
}
int dbg_register(dbg_reader reader) {
    int* n;
    dbg_reader* r = dbg_readers(&n);
    if (*n < 32) r[(*n)++] = reader;
    return *n;
}
int debug_violations(uint64_t* count, int32_t* first_code) {
    if (cudaDeviceSynchronize() != cudaSuccess) return TRON_ERR_CUDA;
    int* n;
    dbg_reader* r = dbg_readers(&n);
    unsigned long long total = 0;
    int first = 0;
    for (int i = 0; i < *n; ++i) {
        unsigned long long c = 0;
        int f = 0;
        if (r[i](&c, &f) != 0) return TRON_ERR_CUDA;
        total += c;
        if (!first && c) first = f;
    }
    if (count) *count = total;
    if (first_code) *first_code = first;
    return TRON_OK;
}
#else
int debug_violations(uint64_t*, int32_t*) { return TRON_ERR_UNSUPPORTED; }
#endif

}  // namespace tron
