// host_env.cu -- host-buffer front end of the C ABI: what a Game.step caller holding numpy arrays binds to.
//
// Per step:  one H2D copy of the actions (+ spawns) on the compute stream; the games are cut into chunks and chunk c's tick kernel is
// followed by an event the COPY stream waits on before it drains that chunk's observations over PCIe, so the D2H stream runs
// back to back behind the kernels; reward / done / winner leave as one whole-array copy each after the last kernel.
// Device observations and scalars are double-buffered: with tron_host_env_step_begin / _wait the kernels of step t+1 run while
// step t is still draining, i.e. the PCIe link (the bound of this path) never idles between steps.
#include <sched.h>
#include <unistd.h>

#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "abi_internal.h"

using namespace tron;

namespace {

// ---- NUMA placement of pinned host memory -----------------------------------------------------------
// cudaHostAlloc takes its pages under the calling thread's memory policy (default: the node of the CPU it runs on), so the
// thread is moved onto the device's local CPUs (sysfs local_cpulist of the PCI function) while the pages are allocated.
bool device_local_cpus(int dev, cpu_set_t* out) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, dev) != cudaSuccess) { cudaGetLastError(); return false; }
    for (char* c = bus; *c; ++c) *c = (char)tolower((unsigned char)*c);
    char path[128];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/local_cpulist", bus);
    FILE* f = fopen(path, "r");
    if (!f) return false;
    char line[4096] = {0};
    const bool got = fgets(line, sizeof line, f) != nullptr;
    fclose(f);
    if (!got) return false;
    CPU_ZERO(out);
    int n_set = 0;
    for (char* tok = strtok(line, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int a = -1, b = -1;
        if (sscanf(tok, "%d-%d", &a, &b) == 2) {}
        else if (sscanf(tok, "%d", &a) == 1) b = a;
        for (int c = a; c >= 0 && c <= b && c < CPU_SETSIZE; ++c) { CPU_SET(c, out); ++n_set; }
    }
    return n_set > 0;
}

struct AffinityNearDevice {  // RAII: narrow the calling thread to (allowed CPUs) n (device-local CPUs)
    cpu_set_t old_set;
    bool moved = false;
    explicit AffinityNearDevice(int dev) {
        cpu_set_t local, both;
        if (sched_getaffinity(0, sizeof old_set, &old_set) != 0 || !device_local_cpus(dev, &local)) return;
        CPU_AND(&both, &old_set, &local);
        if (CPU_COUNT(&both) == 0 || CPU_EQUAL(&both, &old_set)) return;
        moved = sched_setaffinity(0, sizeof both, &both) == 0;
    }
    ~AffinityNearDevice() { if (moved) sched_setaffinity(0, sizeof old_set, &old_set); }
};

}  // namespace

extern "C" {

struct tron_host_env {
    tron_step_args proto;
    int device;
    int n_chunks;
    int planes, cells, esize;
    bool reset_done;
    void* d_state;
    uint8_t* d_actions;
    int8_t* d_spawn;
    void* d_obs[2];       // double-buffered by step parity
    float* d_reward[2];
    uint8_t* d_done[2];
    uint8_t* d_winner[2];
    uint64_t counter;
    uint64_t begun, waited;  // steps enqueued / steps whose outputs have landed
    cudaStream_t compute, copy;
    std::vector<cudaEvent_t> chunk_ready;  // kernel of chunk c finished (per buffer: [2][n_chunks])
    cudaEvent_t scalars_ready[2];          // last kernel of the step finished
    cudaEvent_t drained[2];                // all D2H copies of the step that used buffer b have landed
    cudaEvent_t inputs_consumed;           // the kernels that read d_actions / d_spawn finished
};

static void host_env_free(tron_host_env* e) {
    if (!e) return;
    DeviceGuard guard(e->device);
    if (e->compute) cudaStreamSynchronize(e->compute);
    if (e->copy) cudaStreamSynchronize(e->copy);
    for (cudaEvent_t ev : e->chunk_ready) cudaEventDestroy(ev);
    for (int b = 0; b < 2; ++b) {
        if (e->scalars_ready[b]) cudaEventDestroy(e->scalars_ready[b]);
        if (e->drained[b]) cudaEventDestroy(e->drained[b]);
        cudaFree(e->d_obs[b]); cudaFree(e->d_reward[b]); cudaFree(e->d_done[b]); cudaFree(e->d_winner[b]);
    }
    if (e->inputs_consumed) cudaEventDestroy(e->inputs_consumed);
    if (e->compute) cudaStreamDestroy(e->compute);
    if (e->copy) cudaStreamDestroy(e->copy);
    cudaFree(e->d_state); cudaFree(e->d_actions); cudaFree(e->d_spawn);
    cudaGetLastError();
    delete e;
}

int tron_host_env_create(tron_host_env** out, const tron_step_args* proto, int n_chunks) {
    if (!out || !proto || proto->struct_size != sizeof(tron_step_args)) return TRON_ERR_INVALID;
    if (!geometry_ok(proto->n_envs, proto->width, proto->height)) return TRON_ERR_INVALID;
    if (n_chunks < 1) n_chunks = 1;
    if (n_chunks > proto->n_envs) n_chunks = proto->n_envs;
    if (n_chunks > 256) n_chunks = 256;
    tron_host_env* e = new (std::nothrow) tron_host_env();
    if (!e) return TRON_ERR_INVALID;
    e->proto = *proto;
    e->proto.obs_prev = 0;  // device observations are double-buffered: a buffer never holds the previous tick
    if (cudaGetDevice(&e->device) != cudaSuccess) { cudaGetLastError(); delete e; return TRON_ERR_CUDA; }
    e->n_chunks = n_chunks;
    e->planes = planes_of(proto->obs_enc);
    e->cells = tron_cells_per_env(proto->width, proto->height);
    e->esize = tron_elem(proto->obs_dtype);
    const size_t N = (size_t)proto->n_envs;
    size_t sb = 0;
    if (tron_state_bytes(proto->n_envs, proto->width, proto->height, proto->layout, &sb) != TRON_OK) { delete e; return TRON_ERR_UNSUPPORTED; }
    bool ok = cudaMalloc(&e->d_state, sb) == cudaSuccess && cudaMemset(e->d_state, 0, sb) == cudaSuccess &&
              cudaMalloc((void**)&e->d_actions, N * 2) == cudaSuccess && cudaMalloc((void**)&e->d_spawn, N * 4) == cudaSuccess;
    for (int b = 0; ok && b < 2; ++b) {
        ok = cudaMalloc((void**)&e->d_reward[b], N * 8) == cudaSuccess && cudaMalloc((void**)&e->d_done[b], N) == cudaSuccess &&
             cudaMalloc((void**)&e->d_winner[b], N) == cudaSuccess;
        if (ok && e->planes) ok = cudaMalloc(&e->d_obs[b], N * 2 * e->planes * e->cells * e->esize) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&e->scalars_ready[b], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&e->drained[b], cudaEventDisableTiming) == cudaSuccess;
    }
    ok = ok && cudaEventCreateWithFlags(&e->inputs_consumed, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&e->compute, cudaStreamNonBlocking) == cudaSuccess &&
         cudaStreamCreateWithFlags(&e->copy, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; ok && i < 2 * n_chunks; ++i) {
        cudaEvent_t ev;
        ok = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) == cudaSuccess;
        if (ok) e->chunk_ready.push_back(ev);
    }
    if (!ok) { cudaGetLastError(); host_env_free(e); return TRON_ERR_CUDA; }
    *out = e;
    return TRON_OK;
}

int tron_host_env_destroy(tron_host_env* env) { host_env_free(env); return TRON_OK; }
void* tron_host_env_state(tron_host_env* env) { return env ? env->d_state : nullptr; }

// block until every enqueued step has landed
static int host_env_drain(tron_host_env* e) {
    bool ok = cudaStreamSynchronize(e->compute) == cudaSuccess;
    ok = (cudaStreamSynchronize(e->copy) == cudaSuccess) && ok;
    e->waited = e->begun;
    if (!ok) { cudaGetLastError(); return TRON_ERR_CUDA; }
    return TRON_OK;
}

// enqueue one pass over the chunks; mode MODE_RESET (reset + observe) or MODE_STEP.  Does not block.
static int host_env_enqueue(tron_host_env* e, int mode, const uint8_t* actions_h, const int8_t* spawn_h, void* obs_h, float* reward_h,
                            uint8_t* done_h, uint8_t* winner_h) {
    const int N = e->proto.n_envs, C = e->cells;
    const int b = (int)(e->begun & 1u);
    const size_t frame = (size_t)2 * e->planes * C * e->esize;  // obs bytes per env
    StepParams base;
    tron_step_args a = e->proto;
    a.state = e->d_state; a.obs = e->d_obs[b]; a.actions = e->d_actions; a.action_dtype = TRON_U8;
    a.reward = e->d_reward[b]; a.done = e->d_done[b]; a.winner = e->d_winner[b]; a.ep_len_out = nullptr; a.stats = nullptr;
    a.obs_terminal = nullptr; a.extra = nullptr;
    a.spawn = spawn_h ? e->d_spawn : nullptr; a.counter = e->counter; a.n_ticks = 1;
    int rc = fill_params(&a, mode == MODE_RESET ? MODE_RESET : MODE_STEP, base);
    if (rc != TRON_OK) return rc;
    StepParams obase = base;
    if (mode == MODE_RESET && obs_h && e->planes) {
        rc = fill_params(&a, MODE_OBSERVE, obase);
        if (rc != TRON_OK) return rc;
    }
    bool ok = true;
    // the buffers of parity b were last used two steps ago: their D2H copies must have drained before the kernels overwrite them
    ok = ok && cudaStreamWaitEvent(e->compute, e->drained[b], 0) == cudaSuccess;
    if (mode == MODE_STEP) ok = ok && cudaMemcpyAsync(e->d_actions, actions_h, 2 * (size_t)N, cudaMemcpyHostToDevice, e->compute) == cudaSuccess;
    if (spawn_h) ok = ok && cudaMemcpyAsync(e->d_spawn, spawn_h, 4 * (size_t)N, cudaMemcpyHostToDevice, e->compute) == cudaSuccess;
    const int per = (N + e->n_chunks - 1) / e->n_chunks;
    for (int c = 0; c < e->n_chunks && ok && rc == TRON_OK; ++c) {
        const int lo = c * per, n = (lo + per <= N ? per : N - lo);
        if (n <= 0) break;
        StepParams p;
        slice_params(base, lo, n, p);
        if (mode == MODE_RESET) {
            rc = dispatch(p, MODE_RESET, TRON_I8, TRON_ENC_NONE, e->compute);
            if (rc == TRON_OK && obs_h && e->planes) {
                StepParams q;
                slice_params(obase, lo, n, q);
                rc = dispatch(q, MODE_OBSERVE, e->proto.obs_dtype, e->proto.obs_enc, e->compute);
            }
        } else {
            rc = dispatch(p, MODE_STEP, e->proto.obs_dtype, e->proto.obs_enc, e->compute);
        }
        if (rc != TRON_OK) break;
        if (obs_h && e->planes) {
            cudaEvent_t ev = e->chunk_ready[(size_t)b * e->n_chunks + c];
            ok = ok && cudaEventRecord(ev, e->compute) == cudaSuccess && cudaStreamWaitEvent(e->copy, ev, 0) == cudaSuccess &&
                 cudaMemcpyAsync((char*)obs_h + (size_t)lo * frame, (char*)e->d_obs[b] + (size_t)lo * frame, (size_t)n * frame, cudaMemcpyDeviceToHost,
                                 e->copy) == cudaSuccess;
        }
    }
    if (rc == TRON_OK && ok) {
        ok = ok && cudaEventRecord(e->scalars_ready[b], e->compute) == cudaSuccess && cudaStreamWaitEvent(e->copy, e->scalars_ready[b], 0) == cudaSuccess;
        if (mode == MODE_STEP) {
            if (reward_h) ok = ok && cudaMemcpyAsync(reward_h, e->d_reward[b], 8 * (size_t)N, cudaMemcpyDeviceToHost, e->copy) == cudaSuccess;
            if (done_h) ok = ok && cudaMemcpyAsync(done_h, e->d_done[b], (size_t)N, cudaMemcpyDeviceToHost, e->copy) == cudaSuccess;
            if (winner_h) ok = ok && cudaMemcpyAsync(winner_h, e->d_winner[b], (size_t)N, cudaMemcpyDeviceToHost, e->copy) == cudaSuccess;
        }
        ok = ok && cudaEventRecord(e->drained[b], e->copy) == cudaSuccess;
    }
    e->counter += 1;
    e->begun += 1;
    if (rc != TRON_OK || !ok) {  // leave no stream running behind a failed call
        host_env_drain(e);
        cudaGetLastError();
        return rc != TRON_OK ? rc : TRON_ERR_CUDA;
    }
    return TRON_OK;
}

int tron_host_env_reset(tron_host_env* env, const int8_t* spawn_host, void* obs_host) {
    if (!env) return TRON_ERR_INVALID;
    DeviceGuard guard(env->device);
    if (!guard.ok) return TRON_ERR_CUDA;
    int rc = host_env_drain(env);
    if (rc != TRON_OK) return rc;
    rc = host_env_enqueue(env, MODE_RESET, nullptr, spawn_host, obs_host, nullptr, nullptr, nullptr);
    if (rc != TRON_OK) return rc;
    rc = host_env_drain(env);
    if (rc == TRON_OK) env->reset_done = true;
    return rc;
}

int tron_host_env_step_begin(tron_host_env* env, const uint8_t* actions_host, const int8_t* spawn_host, void* obs_host, float* reward_host,
                             uint8_t* done_host, uint8_t* winner_host) {
    if (!env || !actions_host) return TRON_ERR_INVALID;
    if (!env->reset_done) return TRON_ERR_INVALID;          // a step before the first reset would tick uninitialised games
    if (env->begun - env->waited >= 2) return TRON_ERR_INVALID;  // at most two steps in flight
    DeviceGuard guard(env->device);
    if (!guard.ok) return TRON_ERR_CUDA;
    return host_env_enqueue(env, MODE_STEP, actions_host, spawn_host, obs_host, reward_host, done_host, winner_host);
}

int tron_host_env_step_wait(tron_host_env* env) {
    if (!env || env->waited >= env->begun) return TRON_ERR_INVALID;
    DeviceGuard guard(env->device);
    if (!guard.ok) return TRON_ERR_CUDA;
    const int b = (int)(env->waited & 1u);
    env->waited += 1;
    if (cudaEventSynchronize(env->drained[b]) != cudaSuccess) { cudaGetLastError(); return TRON_ERR_CUDA; }
    return TRON_OK;
}

int tron_host_env_step(tron_host_env* env, const uint8_t* actions_host, const int8_t* spawn_host, void* obs_host, float* reward_host,
                       uint8_t* done_host, uint8_t* winner_host) {
    if (!env) return TRON_ERR_INVALID;
    while (env->waited < env->begun) {
        const int rc = tron_host_env_step_wait(env);
        if (rc != TRON_OK) return rc;
    }
    int rc = tron_host_env_step_begin(env, actions_host, spawn_host, obs_host, reward_host, done_host, winner_host);
    if (rc != TRON_OK) return rc;
    return tron_host_env_step_wait(env);
}

int tron_host_alloc(void** ptr, size_t bytes) {
    if (!ptr || !bytes) return TRON_ERR_INVALID;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return TRON_ERR_CUDA; }
    AffinityNearDevice near(dev);
    if (cudaHostAlloc(ptr, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return TRON_ERR_CUDA; }
    return TRON_OK;
}
int tron_host_free(void* ptr) {
    if (!ptr) return TRON_OK;
    if (cudaFreeHost(ptr) != cudaSuccess) { cudaGetLastError(); return TRON_ERR_CUDA; }
    return TRON_OK;
}

int tron_host_copy_bandwidth(size_t bytes, int direction, int repeats, double* gb_per_s) {
    if (!bytes || !gb_per_s || repeats < 1 || (direction != 0 && direction != 1)) return TRON_ERR_INVALID;
    void* h = nullptr;
    void* d = nullptr;
    cudaStream_t s = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int rc = tron_host_alloc(&h, bytes);
    if (rc != TRON_OK) return rc;
    bool ok = cudaMalloc(&d, bytes) == cudaSuccess && cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess;
    const cudaMemcpyKind kind = direction == 0 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
    void* dst = direction == 0 ? d : h;
    const void* src = direction == 0 ? h : d;
    float ms = 0.f;
    if (ok) {
        memset(h, 1, bytes);
        ok = cudaMemsetAsync(d, 1, bytes, s) == cudaSuccess && cudaMemcpyAsync(dst, src, bytes, kind, s) == cudaSuccess;  // warm-up
        ok = ok && cudaEventRecord(e0, s) == cudaSuccess;
        for (int i = 0; ok && i < repeats; ++i) ok = cudaMemcpyAsync(dst, src, bytes, kind, s) == cudaSuccess;
        ok = ok && cudaEventRecord(e1, s) == cudaSuccess && cudaStreamSynchronize(s) == cudaSuccess && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess;
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (s) cudaStreamDestroy(s);
    cudaFree(d);
    tron_host_free(h);
    if (!ok || ms <= 0.f) { cudaGetLastError(); return TRON_ERR_CUDA; }
    *gb_per_s = (double)bytes * repeats / (ms * 1e-3) / 1e9;
    return TRON_OK;
}

}  // extern "C"
