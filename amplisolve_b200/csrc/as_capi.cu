// C ABI of libamplisolve_b200.so: contexts, the _dev entry points (enqueue on the caller's stream) and
// the _host entry points (slot-tiled, double-buffered H2D -> kernel -> D2H pipelines).
// Interface contract and reference citations: include/amplisolve_b200.h.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <atomic>
#include <cmath>
#include <cstring>
#include <ctime>
#include <cstdlib>
#include <string>
#include <thread>
#include <vector>

#include "as_kernels.h"
#include "as_wire.h"

static thread_local char g_err[512] = "";

// AS_TIMING=1 in the environment: one "AS_TIMING <phase> <seconds>" line per phase of the _host pipelines on stderr
struct PhaseClock {
    bool on;
    double t0;
    static double now() {
        timespec ts;
        clock_gettime(CLOCK_MONOTONIC, &ts);
        return ts.tv_sec + 1e-9 * ts.tv_nsec;
    }
    PhaseClock() : on(getenv("AS_TIMING") != nullptr), t0(now()) {}
    void lap(const char* phase) {
        const double t1 = now();
        if (on) fprintf(stderr, "AS_TIMING capi.%s %.6f\n", phase, t1 - t0);
        t0 = t1;
    }
};

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) return fail(AS_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                                           __FILE__, __LINE__);                                           \
    } while (0)

struct DevBuf {  // grow-only device scratch
    void* p = nullptr;
    size_t bytes = 0;
    cudaError_t need(size_t n) {
        if (n <= bytes) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
        cudaError_t e = cudaMalloc(&p, n);
        if (e == cudaSuccess) bytes = n;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

struct PinnedBuf {  // pinned host scratch, released on every exit path
    void* p = nullptr;
    ~PinnedBuf() { if (p) cudaFreeHost(p); }
    cudaError_t alloc(size_t n) { return cudaHostAlloc(&p, n ? n : 16, cudaHostAllocDefault); }
};

struct PinnedGrow {  // grow-only pinned host scratch owned by the context (cudaHostAlloc costs ~1 ms: not per call)
    void* p = nullptr;
    size_t bytes = 0;
    cudaError_t need(size_t n) {
        if (n <= bytes) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; bytes = 0;
        cudaError_t e = cudaHostAlloc(&p, n, cudaHostAllocDefault);
        if (e == cudaSuccess) bytes = n;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; bytes = 0; }
};

struct as_ctx {
    int device = 0;
    std::vector<as_ctx*> subs;  // as_create_multi: one single-device context per GPU; the _host entry points shard over them
    int call_variant = AS_DEFAULT_CALL_KERNEL;   // 0 straightforward, 1 queued (direct loads), >= 2 TMA-staged (K, stages) variants
    int noise_cfg = AS_DEFAULT_NOISE_KERNEL;      // 0 direct loads, >= 1 TMA-staged (K, stages) variants
    int64_t launches = 0;
    int64_t host_tile_slots = 0;  // 0 = automatic
    int64_t defer_cap_override = 0;  // > 0: capacity of the deferred caller's candidate list (tests of the overflow path)
    int fwd_pending_cap = 0;         // > 0: usable depth of call_forward_kernel's pending ring (tests of its drain path)
    cudaStream_t copy_stream = nullptr, exec_stream = nullptr, aux_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev_up[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    cudaEvent_t ev_chunk[AS_DEFER_MAX_CHUNKS + 1] = {};  // deferred caller: scan of piece i -> resolve / series on aux_stream
    int defer_chunks = 1;  // pieces of the deferred caller (measured 1/2/3/4/8 pieces: 5.79 / 6.17 / 5.91 / 5.99 / 6.54 ms -- the series of one piece does not overlap the scan of the next, whose CTAs hold every SM)
    DevBuf heads, nheads;                         // twin-group scratch of the _dev noise path
    DevBuf tile[2], tile16[2], wide[2], out[2], aux[2], misc, calls, sortbuf;  // _host pipelines
    DevBuf defer;                                                              // candidate / survivor lists of the deferred caller
    DevBuf lgtab;                                                              // lgamma(i + 1), i < lg_n (as_fisher_tests_host)
    DevBuf sites;                                                              // as_site_tests_host*
    PinnedGrow h_sites;
    int64_t lg_n = 0;
    PinnedGrow h_links, h_small;                                              // _host pipelines, host side
    DevBuf pile_first, pile_pos, pile_counts, pile_rec, pile_off, pile_ref, pile_stats;  // as_pileup_*
    DevBuf pile_slots, pile_wire, pile_wide;                                            // as_pileup_end_wire
    int64_t pile_P = -1;
    int32_t pile_contigs = 0;
    double pile_kernel_ms = 0, pile_h2d_ms = 0;  // AS_TIMING only
};

extern "C" {

const char* as_last_error(void) { return g_err; }
const char* as_version(void) { return "amplisolve_b200 0.1 (sm_100a)"; }

int as_device_count(int* n) {
    if (!n) return fail(AS_EINVAL, "n is NULL");
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) { *n = 0; return fail(AS_ECUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
    *n = c;
    return AS_OK;
}

int as_create(int device, as_ctx** out) {
    if (!out) return fail(AS_EINVAL, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(AS_ECUDA, "no CUDA device available (%s): amplisolve_b200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= n) return fail(AS_EINVAL, "device %d out of range (0..%d)", device, n - 1);
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(AS_ECUDA, "device %d is sm_%d%d; this library carries sm_100a code only", device, prop.major,
                    prop.minor);
    CU(cudaSetDevice(device));
    as_ctx* c = new as_ctx();
    c->device = device;
    CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c->exec_stream, cudaStreamNonBlocking));
    {
        // highest priority: its few CTAs must be dispatched between the waves of the streaming kernel, not after them
        int lo = 0, hi = 0;
        CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CU(cudaStreamCreateWithPriority(&c->aux_stream, cudaStreamNonBlocking, hi));
    }
    CU(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
    for (int i = 0; i < 2; ++i) {
        CU(cudaEventCreateWithFlags(&c->ev_up[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming));
    }
    for (int i = 0; i <= AS_DEFER_MAX_CHUNKS; ++i) CU(cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming));
    if (const char* env = getenv("AS_DEFER_CHUNKS")) c->defer_chunks = std::max(1, std::min(AS_DEFER_MAX_CHUNKS, atoi(env)));
    *out = c;
    return AS_OK;
}

// One context over several GPUs of the box: the _host entry points shard the panel's slots over them (contiguous ranges
// that keep twin groups whole, one host thread per device, no data-path exchange between devices) and merge the call
// lists.  _dev entry points and the element-wise evaluators run on the first device.
int as_create_multi(const int* devices, int ndev, as_ctx** out) {
    if (!out) return fail(AS_EINVAL, "out is NULL");
    *out = nullptr;
    if (!devices || ndev < 1 || ndev > AS_MAX_DEVICES) return fail(AS_EINVAL, "as_create_multi takes 1..%d devices", AS_MAX_DEVICES);
    for (int i = 0; i < ndev; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j]) return fail(AS_EINVAL, "device %d listed twice", devices[i]);
    // one thread per device: context creation takes about a second per GPU and the GPUs do not wait for each other
    std::vector<as_ctx*> made((size_t)ndev, nullptr);
    std::vector<int> rcs((size_t)ndev, AS_OK);
    std::vector<std::string> errs((size_t)ndev);
    auto make = [&](int i) {
        rcs[(size_t)i] = as_create(devices[i], &made[(size_t)i]);
        if (rcs[(size_t)i] != AS_OK) errs[(size_t)i] = g_err;
    };
    {
        std::vector<std::thread> th;
        for (int i = 1; i < ndev; ++i) th.emplace_back(make, i);
        make(0);
        for (auto& t : th) t.join();
    }
    for (int i = 0; i < ndev; ++i) {
        if (rcs[(size_t)i] == AS_OK) continue;
        for (int k = 0; k < ndev; ++k) as_destroy(made[(size_t)k]);
        return fail(rcs[(size_t)i], "%s", errs[(size_t)i].c_str());
    }
    as_ctx* head = made[0];
    if (ndev > 1) {
        head->subs = made;
        cudaSetDevice(head->device);
    }
    *out = head;
    return AS_OK;
}

int as_context_devices(const as_ctx* c, int* devices, int cap) {
    if (!c) return 0;
    const int n = c->subs.empty() ? 1 : (int)c->subs.size();
    for (int i = 0; i < n && i < cap && devices; ++i) devices[i] = c->subs.empty() ? c->device : c->subs[(size_t)i]->device;
    return n;
}

void as_destroy(as_ctx* c) {
    if (!c) return;
    for (size_t k = 1; k < c->subs.size(); ++k) as_destroy(c->subs[k]);
    c->subs.clear();
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    c->heads.release(); c->nheads.release(); c->misc.release(); c->calls.release(); c->sortbuf.release();
    c->h_links.release(); c->h_small.release(); c->lgtab.release(); c->defer.release(); c->sites.release(); c->h_sites.release();
    c->pile_first.release(); c->pile_pos.release(); c->pile_counts.release(); c->pile_rec.release(); c->pile_off.release();
    c->pile_ref.release(); c->pile_stats.release(); c->pile_slots.release(); c->pile_wire.release(); c->pile_wide.release();
    for (int i = 0; i < 2; ++i) {
        c->tile[i].release(); c->tile16[i].release(); c->wide[i].release(); c->out[i].release(); c->aux[i].release();
        if (c->ev_up[i]) cudaEventDestroy(c->ev_up[i]);
        if (c->ev_done[i]) cudaEventDestroy(c->ev_done[i]);
    }
    for (int i = 0; i <= AS_DEFER_MAX_CHUNKS; ++i)
        if (c->ev_chunk[i]) cudaEventDestroy(c->ev_chunk[i]);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->exec_stream) cudaStreamDestroy(c->exec_stream);
    delete c;
}

int as_host_alloc(void** out, size_t bytes) {
    if (!out) return fail(AS_EINVAL, "out is NULL");
    CU(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
    return AS_OK;
}
int as_host_free(void* p) {
    CU(cudaFreeHost(p));
    return AS_OK;
}

int as_set_host_tile_slots(as_ctx* c, int64_t slots);
int as_set_call_kernel(as_ctx* c, int variant) {
    if (!c || variant < -1 || variant > 20) return fail(AS_EINVAL, "bad call kernel variant");
    c->call_variant = variant < 0 ? AS_DEFAULT_CALL_KERNEL : variant;
    for (size_t k = 1; k < c->subs.size(); ++k) c->subs[k]->call_variant = c->call_variant;
    return AS_OK;
}
int as_set_noise_kernel(as_ctx* c, int variant) {
    if (!c || variant < -1 || variant > 8) return fail(AS_EINVAL, "bad noise kernel variant");
    c->noise_cfg = variant < 0 ? AS_DEFAULT_NOISE_KERNEL : variant;
    for (size_t k = 1; k < c->subs.size(); ++k) c->subs[k]->noise_cfg = c->noise_cfg;
    return AS_OK;
}
int64_t as_kernel_launches(const as_ctx* c) {
    if (!c) return 0;
    int64_t n = c->launches;
    for (size_t k = 1; k < c->subs.size(); ++k) n += c->subs[k]->launches;
    return n;
}
int as_set_option(as_ctx* c, const char* name, int64_t value) {
    if (!c || !name) return fail(AS_EINVAL, "bad argument");
    if (!strcmp(name, "call_kernel")) return as_set_call_kernel(c, (int)value);
    if (!strcmp(name, "noise_kernel")) return as_set_noise_kernel(c, (int)value);
    if (!strcmp(name, "host_tile_slots")) return as_set_host_tile_slots(c, value);
    if (!strcmp(name, "deferred_chunks")) {
        if (value < 1 || value > AS_DEFER_MAX_CHUNKS) return fail(AS_EINVAL, "deferred_chunks must be 1..%d", AS_DEFER_MAX_CHUNKS);
        c->defer_chunks = (int)value;
        return AS_OK;
    }
    if (!strcmp(name, "forward_pending_cap")) {
        if (value < 0 || value > AS_FWD_PENDING) return fail(AS_EINVAL, "forward_pending_cap must be 0 (automatic) .. %d", AS_FWD_PENDING);
        c->fwd_pending_cap = (int)value;
        for (size_t k = 1; k < c->subs.size(); ++k) c->subs[k]->fwd_pending_cap = (int)value;
        return AS_OK;
    }
    if (!strcmp(name, "deferred_capacity")) {
        if (value < 0) return fail(AS_EINVAL, "deferred_capacity must be >= 0 (0 = automatic)");
        c->defer_cap_override = value;
        return AS_OK;
    }
    return fail(AS_EINVAL, "unknown option %s", name);
}
int as_set_host_tile_slots(as_ctx* c, int64_t slots) {
    if (!c || slots < 0 || (slots % 128) != 0) return fail(AS_EINVAL, "host tile size must be 0 (automatic) or a multiple of 128 slots");
    c->host_tile_slots = slots;
    for (size_t k = 1; k < c->subs.size(); ++k) c->subs[k]->host_tile_slots = slots;
    return AS_OK;
}

static int check_common(as_ctx* c, const void* counts, int32_t n_samples, int64_t P, int64_t b, int64_t e, int32_t cut) {
    if (!c) return fail(AS_EINVAL, "ctx is NULL");
    if (!counts) return fail(AS_EINVAL, "counts is NULL");
    if (((uintptr_t)counts & 15) != 0) return fail(AS_EINVAL, "counts must be 16-byte aligned");
    if (n_samples < 0 || P < 0) return fail(AS_EINVAL, "negative extent");
    if (P > 0x7fffffffll) return fail(AS_EINVAL, "at most 2^31-1 slots per call (shard the panel)");
    if (b < 0 || e > P || b > e) return fail(AS_EINVAL, "bad slot range [%lld,%lld) of %lld", (long long)b, (long long)e, (long long)P);
    if (cut < 1) return fail(AS_EINVAL, "coverage cutoff must be >= 1 (the programs map <= 0 to 100, EE:383, VC:277)");
    return AS_OK;
}

// ---- noise -----------------------------------------------------------------------------------------
int as_noise_estimate_dev(as_ctx* c, const uint32_t* d_counts, int32_t S, int64_t P, int64_t b, int64_t e,
                          const int32_t* d_twin_next, const int32_t* d_twin_head, float C, int32_t cut, float* d_thr,
                          float* d_germ_val, uint8_t* d_germ_state, uint32_t* d_count, uint32_t* d_nrec, void* stream) {
    int rc = check_common(c, d_counts, S, P, b, e, cut);
    if (rc) return rc;
    if (!d_thr || !d_germ_val || !d_germ_state || !d_count || !d_nrec) return fail(AS_EINVAL, "output pointer is NULL");
    if ((d_twin_next == nullptr) != (d_twin_head == nullptr)) return fail(AS_EINVAL, "twin_next and twin_head go together");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (d_twin_next) {
        CU(c->heads.need(sizeof(int32_t) * 2 * (size_t)((e - b + 1) / 2 + 1)));
        CU(c->nheads.need(2 * sizeof(uint32_t)));
        CU(cudaEventRecord(c->ev_fork, st));
    }
    // the streaming kernel goes out first so that it starts at once ...
    CU(as_launch_noise_main(c->noise_cfg, d_counts, S, P, b, e, d_twin_next, d_twin_head, 0, C, (uint32_t)cut, d_thr, d_germ_val,
                            d_germ_state, d_count, d_nrec, st));
    c->launches += 1;
    if (d_twin_next) {
        // ... and the twin groups it leaves out (pairs cut by a CTA tile, longer chains: scattered reads, a few CTAs)
        // run beside it on a second stream; they write other slots.  Joined before control returns to the caller's stream.
        CU(cudaStreamWaitEvent(c->aux_stream, c->ev_fork, 0));
        CU(as_launch_noise_twins(c->noise_cfg, d_counts, S, P, b, e, d_twin_next, d_twin_head, (int32_t*)c->heads.p,
                                 (uint32_t*)c->nheads.p, C, (uint32_t)cut, d_thr, d_germ_val, d_germ_state, d_count,
                                 d_nrec, c->aux_stream));
        CU(cudaEventRecord(c->ev_join, c->aux_stream));
        c->launches += 3;
        CU(cudaStreamWaitEvent(st, c->ev_join, 0));
    }
    return AS_OK;
}

int as_noise_estimate_sweep_dev(as_ctx* c, const uint32_t* d_counts, int32_t S, int64_t P, int64_t b, int64_t e,
                                const int32_t* d_twin_next, const int32_t* d_twin_head, const float* c_values, int32_t n_c,
                                int32_t cut, float* d_thr, float* d_germ_val, uint8_t* d_germ_state, uint32_t* d_count,
                                uint32_t* d_nrec, void* stream) {
    if (!c_values || n_c < 1 || n_c > 8) return fail(AS_EINVAL, "a sweep takes 1..8 values of C");
    int rc = check_common(c, d_counts, S, P, b, e, cut);
    if (rc) return rc;
    if (!d_thr || !d_germ_val || !d_germ_state || !d_count || !d_nrec) return fail(AS_EINVAL, "output pointer is NULL");
    if ((d_twin_next == nullptr) != (d_twin_head == nullptr)) return fail(AS_EINVAL, "twin_next and twin_head go together");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t stride = P * 8;
    if (d_twin_next) {
        CU(c->heads.need(sizeof(int32_t) * 2 * (size_t)((e - b + 1) / 2 + 1)));
        CU(c->nheads.need(2 * sizeof(uint32_t)));
        CU(cudaEventRecord(c->ev_fork, st));
    }
    // ONE pass over the normals for all values (noise_pattern_kernel): every output, in-tile twin pairs included
    const int geom = c->noise_cfg >= 7 ? c->noise_cfg - 7 : 0;
    CU(as_launch_noise_pattern(geom, d_counts, S, P, b, e, d_twin_next, d_twin_head, 0, c_values, n_c, (uint32_t)cut, d_thr, stride,
                               d_germ_val, d_germ_state, d_count, d_nrec, st));
    c->launches += 1;
    if (d_twin_next) {
        // the twin groups it leaves out (pairs cut by a CTA tile, longer chains: a few slots, scattered reads) run beside it
        // on the side stream, value by value; they rewrite Germ_Max / count / nrec of those slots with the same values
        CU(cudaStreamWaitEvent(c->aux_stream, c->ev_fork, 0));
        CU(as_launch_twin_heads(7, b, e, d_twin_next, d_twin_head, (int32_t*)c->heads.p, (uint32_t*)c->nheads.p, c->aux_stream));
        c->launches += 1;
        for (int32_t i = 0; i < n_c; ++i) {
            CU(as_launch_noise_twin_groups(d_counts, S, P, b, e, d_twin_next, (const int32_t*)c->heads.p, (const uint32_t*)c->nheads.p,
                                           c_values[i], (uint32_t)cut, d_thr + (int64_t)i * stride, d_germ_val, d_germ_state, d_count,
                                           d_nrec, c->aux_stream));
            c->launches += 2;
        }
        CU(cudaEventRecord(c->ev_join, c->aux_stream));
        CU(cudaStreamWaitEvent(st, c->ev_join, 0));
    }
    return AS_OK;
}

int as_thresholds_caller_view_dev(as_ctx* c, const float* d_thr, float* d_view, int64_t n, void* stream) {
    if (!c || !d_thr || !d_view || n < 0) return fail(AS_EINVAL, "bad argument");
    CU(cudaSetDevice(c->device));
    CU(as_launch_thr_view(d_thr, d_view, n, (cudaStream_t)stream));
    c->launches += 1;
    return AS_OK;
}

// Slots per tile of the _host pipelines: ~256 MiB of host data per buffer (elem * 8 bytes per record: the denser the
// host format, the more slots per tile and the fewer tiles), multiple of 1024 slots.
#define AS_HOST_TILE_MB_DEFAULT 256
static int64_t tile_slots(const as_ctx* c, int32_t n_samples, int64_t P, int elem) {
    if (c->host_tile_slots > 0) return std::min(c->host_tile_slots, std::max<int64_t>(P, 1));
    const int64_t per_slot = 8ll * elem * std::max(1, n_samples);
    static const int64_t tile_mb = []() {  // host bytes per upload tile; AS_HOST_TILE_MB overrides (measurements)
        const char* env = getenv("AS_HOST_TILE_MB");
        const long v = env ? atol(env) : 0;
        return (int64_t)(v > 0 ? v : AS_HOST_TILE_MB_DEFAULT);
    }();
    int64_t t = (tile_mb << 20) / per_slot;
    t = std::max<int64_t>(1024, (t / 1024) * 1024);
    return std::min(t, std::max<int64_t>(P, 1));
}

// A host count tensor: uint32 (elem = 4), the uint16 wire format (elem = 2) or the packed wire format (elem = 1: one
// uint32 per (sample, strand, slot)); the two wire formats come with a side list of wide records.  elem * 4 = bytes per
// (sample, strand, slot).
struct HostSrc {
    const void* counts;
    int elem;
    const as_wide_record* wide;  // sorted by slot
    int64_t n_wide;
};

// upload slots [p0, p0+n) of a host tensor [n_samples][2][P][4] into a packed device tile [n_samples][2][n][4] of uint32.
// elem = 4: the host tensor is uint32.  elem = 2 / 1: it is in a wire format; the smaller tile goes through a staging
// buffer and is widened / unpacked on the device, then the escaped records of the tile are patched in.
static cudaError_t upload_tile(as_ctx* c, int bsel, const HostSrc& src, int32_t n_samples, int64_t P, int64_t p0, int64_t n,
                               cudaStream_t st) {
    const size_t word = (size_t)src.elem * 4;  // bytes per (sample, strand, slot)
    void* dst = src.elem == 4 ? c->tile[bsel].p : c->tile16[bsel].p;
    return cudaMemcpy2DAsync(dst, (size_t)n * word, (const char*)src.counts + (size_t)p0 * word, (size_t)P * word,
                             (size_t)n * word, (size_t)n_samples * 2, cudaMemcpyHostToDevice, st);
}

// wire formats: the uploaded tile is widened / unpacked into the uint32 tile and the escaped records of the tile are
// patched in from the device copy of the side list.  Runs on the EXEC stream (after the upload event), so that the copy
// stream goes straight on to the next tile.
static cudaError_t expand_tile(as_ctx* c, int bsel, const HostSrc& src, int32_t n_samples, int64_t p0, int64_t n, cudaStream_t st) {
    if (src.elem == 4) return cudaSuccess;
    const void* stg = c->tile16[bsel].p;
    cudaError_t e = src.elem == 2 ? as_launch_widen16((const uint16_t*)stg, (uint32_t*)c->tile[bsel].p, (int64_t)n_samples * 2 * n, st)
                                  : as_launch_unpack((const uint32_t*)stg, (uint32_t*)c->tile[bsel].p, (int64_t)n_samples * 2 * n, st);
    c->launches += 1;
    if (e != cudaSuccess || src.n_wide == 0) return e;
    const as_wide_record* lo = std::lower_bound(src.wide, src.wide + src.n_wide, p0,
                                                [](const as_wide_record& r, int64_t v) { return (int64_t)r.slot < v; });
    const as_wide_record* hi = std::lower_bound(lo, src.wide + src.n_wide, p0 + n,
                                                [](const as_wide_record& r, int64_t v) { return (int64_t)r.slot < v; });
    const int64_t m = hi - lo;
    if (m == 0) return e;
    c->launches += 1;  // the whole list is on the device already (stage_wide)
    return as_launch_patch_wide((const as_wide_record*)c->wide[0].p + (lo - src.wide), m, (uint32_t*)c->tile[bsel].p, n, p0,
                                n_samples, st);
}

// the side list of a wire-format tensor goes to the device once, ahead of the first tile, on the stream the tiles are
// uploaded on (one copy instead of one small pageable copy per tile, which would stall the upload queue every tile)
static cudaError_t stage_wide(as_ctx* c, const HostSrc& src, cudaStream_t st) {
    if (src.elem == 4 || src.n_wide == 0) return cudaSuccess;
    cudaError_t e = c->wide[0].need((size_t)src.n_wide * sizeof(as_wide_record));
    if (e != cudaSuccess) return e;
    return cudaMemcpyAsync(c->wide[0].p, src.wide, (size_t)src.n_wide * sizeof(as_wide_record), cudaMemcpyHostToDevice, st);
}

// the eight counts of (sample, slot) out of a host tensor in either format (used for the few gathered twin members)
static void host_record(const HostSrc& src, int64_t P, int64_t sample, int64_t slot, uint32_t* fw, uint32_t* bw) {
    const int64_t wf = (sample * 2) * P + slot, wb = wf + P;
    if (src.elem == 4) {
        memcpy(fw, (const uint32_t*)src.counts + wf * 4, 16);
        memcpy(bw, (const uint32_t*)src.counts + wb * 4, 16);
        return;
    }
    bool absent, escaped;
    if (src.elem == 2) {
        const uint16_t* f = (const uint16_t*)src.counts + wf * 4;
        absent = f[0] == AS_WIRE_ABSENT;
        escaped = f[0] == AS_WIRE_ESCAPE;
    } else {
        const uint32_t w = ((const uint32_t*)src.counts)[wf];
        absent = w == AS_PACKED_ABSENT;
        escaped = w == AS_PACKED_ESCAPE;
    }
    if (absent) {
        for (int i = 0; i < 4; ++i) fw[i] = bw[i] = AS_ABSENT;
    } else if (escaped) {  // the real counts are in the side list
        const as_wide_record* r = std::lower_bound(src.wide, src.wide + src.n_wide, slot,
                                                   [](const as_wide_record& x, int64_t v) { return (int64_t)x.slot < v; });
        for (; r < src.wide + src.n_wide && r->slot == slot; ++r)
            if (r->sample == sample) { memcpy(fw, r->fw, 16); memcpy(bw, r->bw, 16); return; }
        for (int i = 0; i < 4; ++i) fw[i] = bw[i] = AS_ABSENT;  // inconsistent input: treated as absent
    } else if (src.elem == 2) {
        const uint16_t* f = (const uint16_t*)src.counts + wf * 4;
        const uint16_t* b = (const uint16_t*)src.counts + wb * 4;
        for (int i = 0; i < 4; ++i) { fw[i] = f[i]; bw[i] = b[i]; }
    } else {
        as_unpack_word(((const uint32_t*)src.counts)[wf], fw);
        as_unpack_word(((const uint32_t*)src.counts)[wb], bw);
    }
}

static int check_wide(const HostSrc& src, int32_t n_samples, int64_t P) {
    if (src.elem == 4) return AS_OK;
    if (src.n_wide < 0 || (src.n_wide > 0 && !src.wide)) return fail(AS_EINVAL, "bad wide-record list");
    // range and order of every record (the tiles find their records by binary search); a few threads for long lists
    const int64_t n = src.n_wide;
    const int nth = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(std::thread::hardware_concurrency(), 16u), n / 100000));
    std::vector<int64_t> bad((size_t)nth, -1);
    auto work = [&](int k) {
        const int64_t lo = n * k / nth, hi = n * (k + 1) / nth;
        for (int64_t i = lo; i < hi; ++i) {
            const as_wide_record& r = src.wide[i];
            if (r.slot < 0 || r.slot >= P || r.sample < 0 || r.sample >= n_samples || (i > 0 && src.wide[i - 1].slot > r.slot)) {
                bad[(size_t)k] = i;
                return;
            }
        }
    };
    std::vector<std::thread> th;
    for (int k = 1; k < nth; ++k) th.emplace_back(work, k);
    work(0);
    for (auto& x : th) x.join();
    for (int k = 0; k < nth; ++k)
        if (bad[(size_t)k] >= 0) return fail(AS_EINVAL, "wide record %lld out of range or out of order (sort by slot)", (long long)bad[(size_t)k]);
    return AS_OK;
}

struct NoiseOutLayout {  // one device block per tile: thr [n_c][n] | germ_val | count | nrec | germ_state | thr_view [n_c][n]
    size_t thr, germ_val, count, nrec, germ_state, view, total;
    NoiseOutLayout(int64_t n, int32_t n_c) {
        thr = 0;
        germ_val = thr + (size_t)n_c * (size_t)n * 32;
        count = germ_val + (size_t)n * 16;
        nrec = count + (size_t)n * 16;
        germ_state = nrec + (size_t)n * 4;
        view = germ_state + (size_t)n * 4;
        total = view + (size_t)n_c * (size_t)n * 32;
    }
};

// Slots [B, E) of the panel on ONE device (c is a single-device context).  Twin groups must not straddle B or E.
// n_c values of C (1..8): thr and thr_view are [n_c][P][4][2].  n_c == 1 runs the single-value kernels (the staged
// streaming kernel is faster than the pattern kernel for one C); n_c > 1 runs noise_pattern_kernel once per tile and
// the twin groups once per value, as as_noise_estimate_sweep_dev does.
static int noise_estimate_host_range(as_ctx* c, const HostSrc& src, int32_t S, int64_t P, int64_t B, int64_t E,
                                     const int32_t* twin_next, const int32_t* twin_head, const float* c_values, int32_t n_c,
                                     int32_t cut, float* thr, float* germ_val, uint8_t* germ_state, uint32_t* count,
                                     uint32_t* nrec, float* thr_view) {
    const int elem = src.elem;
    PhaseClock clk;
    if (E <= B) return AS_OK;
    CU(cudaSetDevice(c->device));
    const int64_t TP = tile_slots(c, S, E - B, elem);
    const NoiseOutLayout lay(TP, n_c);
    for (int i = 0; i < 2; ++i) {
        CU(c->tile[i].need((size_t)TP * 32 * (size_t)std::max(1, S)));
        if (elem != 4) CU(c->tile16[i].need((size_t)TP * 8 * (size_t)elem * (size_t)std::max(1, S)));
        CU(c->out[i].need(lay.total));
        if (twin_next) CU(c->aux[i].need((size_t)TP * 8));
    }
    // pass 1, tile by tile (the copy of tile i+1 overlaps the kernels of tile i): singleton slots by the streaming
    // kernel, twin groups that lie completely inside the tile by the twin kernels on tile-local links.  A group that
    // straddles a tile boundary is excluded here (all its members get head = -1) and done in pass 2.
    int64_t ntiles = (E - B + TP - 1) / TP;
    int32_t* h_links = nullptr;     // pinned: the tile-local links of every tile, tile at p0 at [2 * (p0 - B), ...): next[n] | head[n]
    std::vector<int32_t> crossing;  // heads of the groups that straddle tiles
    if (twin_next) {
        CU(c->h_links.need((size_t)(E - B) * 8));
        h_links = (int32_t*)c->h_links.p;
        CU(c->heads.need(sizeof(int32_t) * 2 * (size_t)((TP + 1) / 2 + 1)));
        CU(c->nheads.need(2 * sizeof(uint32_t)));
        // every slot's verdict depends on its own chain only (does the whole group lie inside the slot's tile?), so
        // the links of all tiles are written by a few threads before the first upload
        const int nth = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(std::thread::hardware_concurrency(), 16u), (E - B) / 65536));
        std::vector<std::vector<int32_t>> cross_t((size_t)nth);
        auto work = [&](int k) {
            for (int64_t g = B + (E - B) * k / nth, ge = B + (E - B) * (k + 1) / nth; g < ge; ++g) {
                const int64_t p0 = B + ((g - B) / TP) * TP, n = std::min(TP, E - p0), i = g - p0;
                int32_t* ln = h_links + (p0 - B) * 2;
                int32_t* lh = ln + n;
                const int64_t h = twin_head[g], nx = twin_next[g];
                if (h == g && nx < 0) { ln[i] = -1; lh[i] = (int32_t)i; continue; }  // singleton
                bool inside = h >= p0 && h <= g;
                if (inside) {
                    int64_t steps = 0;
                    for (int64_t q = h; q >= 0; q = twin_next[q])
                        if (q < p0 || q >= p0 + n || ++steps > n) { inside = false; break; }  // leaves the tile (or malformed: pass 2 reports it)
                }
                if (inside) {
                    ln[i] = nx >= 0 ? (int32_t)(nx - p0) : -1;
                    lh[i] = (int32_t)(h - p0);
                } else {
                    ln[i] = -1;
                    lh[i] = -1;  // neither a singleton nor a head: skipped by every tile kernel
                    if (h == g) cross_t[(size_t)k].push_back((int32_t)g);
                }
            }
        };
        std::vector<std::thread> th;
        for (int k = 1; k < nth; ++k) th.emplace_back(work, k);
        work(0);
        for (auto& x : th) x.join();
        for (const auto& v : cross_t) crossing.insert(crossing.end(), v.begin(), v.end());  // ascending: the chunks are
    }
    clk.lap("noise.checks_alloc");
    CU(stage_wide(c, src, c->copy_stream));
    clk.lap("noise.stage_wide");
    int ret1 = AS_OK;
#define CUT(call) { cudaError_t e_ = (call); if (e_ != cudaSuccess) { ret1 = fail(AS_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); break; } }
    for (int64_t t = 0; t < ntiles; ++t) {
        const int bsel = (int)(t & 1);
        const int64_t p0 = B + t * TP, n = std::min(TP, E - p0);
        if (t >= 2) CUT(cudaStreamWaitEvent(c->copy_stream, c->ev_done[bsel], 0));  // buffer free again
        CUT(upload_tile(c, bsel, src, S, P, p0, n, c->copy_stream));
        int32_t *d_tn = nullptr, *d_th = nullptr;
        if (twin_next) {
            d_tn = (int32_t*)c->aux[bsel].p;
            d_th = d_tn + n;
            CUT(cudaMemcpyAsync(d_tn, h_links + (p0 - B) * 2, (size_t)n * 8, cudaMemcpyHostToDevice, c->copy_stream));
        }
        CUT(cudaEventRecord(c->ev_up[bsel], c->copy_stream));
        CUT(cudaStreamWaitEvent(c->exec_stream, c->ev_up[bsel], 0));
        CUT(expand_tile(c, bsel, src, S, p0, n, c->exec_stream));
        char* o = (char*)c->out[bsel].p;
        if (twin_next) CUT(cudaMemsetAsync(o, 0, lay.total, c->exec_stream));  // slots of crossing groups are filled in pass 2
        float* o_thr = (float*)(o + lay.thr);
        float* o_gv = (float*)(o + lay.germ_val);
        uint8_t* o_gs = (uint8_t*)(o + lay.germ_state);
        uint32_t* o_cnt = (uint32_t*)(o + lay.count);
        uint32_t* o_nrec = (uint32_t*)(o + lay.nrec);
        const uint32_t* d_tile = (const uint32_t*)c->tile[bsel].p;
        // table i of the tile at o_thr + i * TP * 8 (the layout's stride), downloaded to thr + i * P * 8
        const int64_t tstride = TP * 8;
        if (n_c == 1) {
            CUT(as_launch_noise_main(c->noise_cfg, d_tile, S, n, 0, n, d_tn, d_th, 0, c_values[0], (uint32_t)cut, o_thr, o_gv, o_gs,
                                     o_cnt, o_nrec, c->exec_stream));
            c->launches += 1;
            if (twin_next) {
                CUT(as_launch_noise_twins(c->noise_cfg, d_tile, S, n, 0, n, d_tn, d_th, (int32_t*)c->heads.p, (uint32_t*)c->nheads.p,
                                          c_values[0], (uint32_t)cut, o_thr, o_gv, o_gs, o_cnt, o_nrec, c->exec_stream));
                c->launches += 3;
            }
        } else {
            const int geom = c->noise_cfg >= 7 ? c->noise_cfg - 7 : 0;
            CUT(as_launch_noise_pattern(geom, d_tile, S, n, 0, n, d_tn, d_th, 0, c_values, n_c, (uint32_t)cut, o_thr, tstride, o_gv,
                                        o_gs, o_cnt, o_nrec, c->exec_stream));
            c->launches += 1;
            if (twin_next) {  // the groups the pattern kernel leaves out (pairs cut by a CTA tile, longer chains), value by value
                CUT(as_launch_twin_heads(7, 0, n, d_tn, d_th, (int32_t*)c->heads.p, (uint32_t*)c->nheads.p, c->exec_stream));
                c->launches += 1;
                for (int32_t i = 0; i < n_c; ++i) {
                    CUT(as_launch_noise_twin_groups(d_tile, S, n, 0, n, d_tn, (const int32_t*)c->heads.p, (const uint32_t*)c->nheads.p,
                                                    c_values[i], (uint32_t)cut, o_thr + i * tstride, o_gv, o_gs, o_cnt, o_nrec,
                                                    c->exec_stream));
                    c->launches += 2;
                }
                if (ret1 != AS_OK) break;
            }
        }
        CUT(cudaMemcpy2DAsync(thr + p0 * 8, (size_t)P * 32, o + lay.thr, (size_t)tstride * 4, (size_t)n * 32, (size_t)n_c,
                              cudaMemcpyDeviceToHost, c->exec_stream));
        CUT(cudaMemcpyAsync(germ_val + p0 * 4, o + lay.germ_val, (size_t)n * 16, cudaMemcpyDeviceToHost, c->exec_stream));
        CUT(cudaMemcpyAsync(count + p0 * 4, o + lay.count, (size_t)n * 16, cudaMemcpyDeviceToHost, c->exec_stream));
        CUT(cudaMemcpyAsync(nrec + p0, o + lay.nrec, (size_t)n * 4, cudaMemcpyDeviceToHost, c->exec_stream));
        CUT(cudaMemcpyAsync(germ_state + p0 * 4, o + lay.germ_state, (size_t)n * 4, cudaMemcpyDeviceToHost, c->exec_stream));
        if (thr_view) {  // the "%f" hand-over of the thresholds, while they are still on the device
            CUT(as_launch_thr_view(o_thr, (float*)(o + lay.view), (n_c - 1) * tstride + n * 8, c->exec_stream));
            c->launches += 1;
            CUT(cudaMemcpy2DAsync(thr_view + p0 * 8, (size_t)P * 32, o + lay.view, (size_t)tstride * 4, (size_t)n * 32, (size_t)n_c,
                                  cudaMemcpyDeviceToHost, c->exec_stream));
        }
        CUT(cudaEventRecord(c->ev_done[bsel], c->exec_stream));
    }
#undef CUT
    clk.lap("noise.enqueue");
    {
        cudaError_t e1 = cudaStreamSynchronize(c->exec_stream), e2 = cudaStreamSynchronize(c->copy_stream);
        clk.lap("noise.drain");
        if (ret1 != AS_OK) return ret1;
        if (e1 != cudaSuccess || e2 != cudaSuccess)
            return fail(AS_ECUDA, "noise pipeline failed: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
    }
    if (!twin_next || crossing.empty()) return AS_OK;

    // pass 2: the few twin groups whose members lie in different tiles.  Their records are gathered (pure data
    // movement) into one compact tensor [S][2][M][4] with compact twin links.
    std::vector<int32_t> members;  // compact id -> panel slot
    std::vector<int32_t> c_next, c_head;
    for (const int32_t p : crossing) {
        {
            const int32_t head_c = (int32_t)members.size();
            for (int32_t q = (int32_t)p; q >= 0; q = twin_next[q]) {
                if (q >= P) return fail(AS_EINVAL, "twin_next[%d] out of range", q);
                members.push_back(q);
                c_head.push_back(head_c);
                c_next.push_back(twin_next[q] >= 0 ? (int32_t)members.size() : -1);
                if ((int64_t)members.size() > P) return fail(AS_EINVAL, "twin_next contains a cycle");
            }
        }
    }
    const int64_t M = (int64_t)members.size();
    if (M == 0) return AS_OK;
    PinnedBuf gather_buf;
    CU(gather_buf.alloc((size_t)M * 32 * (size_t)std::max(1, S)));
    uint32_t* h_gather = (uint32_t*)gather_buf.p;
    for (int64_t smp = 0; smp < S; ++smp)
        for (int64_t m = 0; m < M; ++m)
            host_record(src, P, smp, members[m], h_gather + ((smp * 2) * M + m) * 4, h_gather + ((smp * 2 + 1) * M + m) * 4);
    const NoiseOutLayout ml(M, n_c);
    DevBuf d_cnt, d_out, d_links;
    cudaError_t e1 = d_cnt.need((size_t)M * 32 * (size_t)std::max(1, S));
    cudaError_t e2 = d_out.need(ml.total);
    cudaError_t e3 = d_links.need((size_t)M * 16 + 64);
    std::vector<char> h_out(ml.total);
    int ret = AS_OK;
    do {
        if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) { ret = fail(AS_ENOMEM, "cudaMalloc failed for the twin tensor"); break; }
        int32_t* d_next = (int32_t*)d_links.p;
        int32_t* d_head = d_next + M;
        int32_t* d_heads = d_head + M;
        cudaStream_t st = c->exec_stream;
#define CUB(call) { cudaError_t e_ = (call); if (e_ != cudaSuccess) { ret = fail(AS_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); break; } }
        CUB(c->nheads.need(2 * sizeof(uint32_t)));
        CUB(cudaMemcpyAsync(d_cnt.p, h_gather, (size_t)M * 32 * (size_t)S, cudaMemcpyHostToDevice, st));
        CUB(cudaMemcpyAsync(d_next, c_next.data(), (size_t)M * 4, cudaMemcpyHostToDevice, st));
        CUB(cudaMemcpyAsync(d_head, c_head.data(), (size_t)M * 4, cudaMemcpyHostToDevice, st));
        char* o = (char*)d_out.p;
        for (int32_t i = 0; i < n_c; ++i) {  // once per value; the C-independent outputs are rewritten with the same values
            CUB(as_launch_noise_twins(0, (const uint32_t*)d_cnt.p, S, M, 0, M, d_next, d_head, d_heads, (uint32_t*)c->nheads.p,
                                      c_values[i], (uint32_t)cut, (float*)(o + ml.thr) + i * M * 8, (float*)(o + ml.germ_val),
                                      (uint8_t*)(o + ml.germ_state), (uint32_t*)(o + ml.count), (uint32_t*)(o + ml.nrec), st));
            c->launches += 3;
        }
        if (ret != AS_OK) break;
        CUB(as_launch_thr_view((float*)(o + ml.thr), (float*)(o + ml.view), n_c * M * 8, st));
        c->launches += 1;
        CUB(cudaMemcpyAsync(h_out.data(), o, ml.total, cudaMemcpyDeviceToHost, st));
        CUB(cudaStreamSynchronize(st));
#undef CUB
        for (int64_t m = 0; m < M; ++m) {
            const int64_t p = members[m];
            for (int64_t i = 0; i < n_c; ++i) {
                memcpy(thr + (i * P + p) * 8, h_out.data() + ml.thr + (i * M + m) * 32, 32);
                if (thr_view) memcpy(thr_view + (i * P + p) * 8, h_out.data() + ml.view + (i * M + m) * 32, 32);
            }
            memcpy(germ_val + p * 4, h_out.data() + ml.germ_val + m * 16, 16);
            memcpy(count + p * 4, h_out.data() + ml.count + m * 16, 16);
            memcpy(nrec + p, h_out.data() + ml.nrec + m * 4, 4);
            memcpy(germ_state + p * 4, h_out.data() + ml.germ_state + m * 4, 4);
        }
    } while (0);
    d_cnt.release(); d_out.release(); d_links.release();
    return ret;
}

// ---- caller ----------------------------------------------------------------------------------------
// the caller as scan -> resolve -> series kernels (as_call_deferred.cu), lists in scratch owned by the context
static int call_deferred(as_ctx* c, const uint32_t* d_counts, int32_t T, int64_t P, int64_t b, int64_t e, const uint8_t* d_ref,
                         const float* d_thr_views, int32_t n_c, int64_t c_stride, int32_t cut, as_call* d_calls, int64_t cap,
                         unsigned long long* d_n_calls, cudaStream_t st) {
    int64_t cap_cand = 0, cap_surv = 0;
    const size_t bytes = as_deferred_scratch_bytes(T, e - b, c->defer_cap_override, &cap_cand, &cap_surv) + 256;
    CU(c->defer.need(bytes));
    CU(as_launch_call_deferred(d_counts, T, P, b, e, d_ref, d_thr_views, n_c, c_stride, (uint32_t)cut, d_calls, cap, d_n_calls, c->defer.p,
                               cap_cand, cap_surv, st, c->aux_stream, c->ev_chunk, c->defer_chunks));
    c->launches += 3 * as_deferred_chunks(e - b, c->defer_chunks);
    return AS_OK;
}

int as_call_variants_dev(as_ctx* c, const uint32_t* d_counts, int32_t T, int64_t P, int64_t b, int64_t e,
                         const uint8_t* d_ref, const float* d_thr_view, int32_t cut, as_call* d_calls, int64_t cap,
                         unsigned long long* d_n_calls, void* stream) {
    int rc = check_common(c, d_counts, T, P, b, e, cut);
    if (rc) return rc;
    if (!d_ref || !d_thr_view || !d_n_calls || (!d_calls && cap > 0) || cap < 0) return fail(AS_EINVAL, "bad pointer / cap");
    if (T >= (1 << 27)) return fail(AS_EINVAL, "at most 2^27-1 samples per call");
    CU(cudaSetDevice(c->device));
    if (c->call_variant == AS_DEFERRED_CALL_KERNEL)
        return call_deferred(c, d_counts, T, P, b, e, d_ref, d_thr_view, 1, P * 8, cut, d_calls, cap, d_n_calls, (cudaStream_t)stream);
    CU(as_launch_call(c->call_variant, d_counts, T, P, b, e, d_ref, d_thr_view, (uint32_t)cut, d_calls, cap, d_n_calls,
                      c->fwd_pending_cap, (cudaStream_t)stream));
    c->launches += 1;
    return AS_OK;
}

int as_call_variants_sweep_dev(as_ctx* c, const uint32_t* d_counts, int32_t T, int64_t P, int64_t b, int64_t e,
                               const uint8_t* d_ref, const float* d_thr_views, int32_t n_c, int32_t cut, as_call* d_calls,
                               int64_t cap, unsigned long long* d_n_calls, void* stream) {
    int rc = check_common(c, d_counts, T, P, b, e, cut);
    if (rc) return rc;
    if (!d_ref || !d_thr_views || !d_n_calls || (!d_calls && cap > 0) || cap < 0) return fail(AS_EINVAL, "bad pointer / cap");
    if (n_c < 1 || n_c > 8) return fail(AS_EINVAL, "a sweep takes 1..8 threshold tables");
    if (T >= (1 << 27)) return fail(AS_EINVAL, "at most 2^27-1 samples per call");
    if (c->call_variant < 2 && n_c > 1) return fail(AS_EINVAL, "the sweep needs a TMA-staged caller variant (>= 2)");
    CU(cudaSetDevice(c->device));
    // default: the deferred pipeline; a staged variant selected by hand runs the in-stage sweep kernel (cross-check)
    if (c->call_variant == AS_DEFERRED_CALL_KERNEL || (c->call_variant == AS_DEFAULT_CALL_KERNEL && n_c > 1))
        return call_deferred(c, d_counts, T, P, b, e, d_ref, d_thr_views, n_c, P * 8, cut, d_calls, cap, d_n_calls, (cudaStream_t)stream);
    CU(as_launch_call_sweep(c->call_variant, d_counts, T, P, b, e, d_ref, d_thr_views, n_c, P * 8, (uint32_t)cut, d_calls, cap,
                            d_n_calls, c->fwd_pending_cap, (cudaStream_t)stream));
    c->launches += 1;
    return AS_OK;
}

// Slots [B, E) of the panel on ONE device (c is a single-device context).  n_c threshold tables (1..8), thr_views
// [n_c][P][4][2].  The calls stay on the device, unsorted, with panel slot ids, in c->calls: list i at i * cap;
// found[i] = the number found for table i (may exceed cap).  n_c == 1 runs the single-table kernel; n_c > 1 runs the
// kernel as_call_variants_sweep_dev would choose (the deferred pipeline by default, the in-stage sweep kernel when a
// staged variant is selected).
static int call_variants_host_range(as_ctx* c, const HostSrc& src, int32_t T, int64_t P, int64_t B, int64_t E, const uint8_t* ref,
                                    const float* thr_views, int32_t n_c, int32_t cut, int64_t cap, int64_t* found) {
    const int elem = src.elem;
    PhaseClock clk;
    for (int32_t i = 0; i < n_c; ++i) found[i] = 0;
    if (E <= B || T == 0) return AS_OK;
    CU(cudaSetDevice(c->device));
    const int64_t TP = tile_slots(c, T, E - B, elem);
    for (int i = 0; i < 2; ++i) {
        CU(c->tile[i].need((size_t)TP * 32 * (size_t)T));
        if (elem != 4) CU(c->tile16[i].need((size_t)TP * 8 * (size_t)elem * (size_t)T));
    }
    // thresholds (n_c * 32 B/slot) and reference bases (1 B/slot) of the range go up once, ahead of the first tile: a
    // per-tile copy from pageable memory would stall the upload queue at every tile.  Table i at d_tv_all + i * (E - B) * 8.
    const int64_t c_stride = (E - B) * 8;
    CU(c->aux[0].need((size_t)(E - B) * (32 * (size_t)n_c + 1) + 64));
    float* d_tv_all = (float*)c->aux[0].p;
    uint8_t* d_rf_all = (uint8_t*)c->aux[0].p + (size_t)(E - B) * 32 * (size_t)n_c;
    CU(cudaMemcpy2DAsync(d_tv_all, (size_t)(E - B) * 32, thr_views + B * 8, (size_t)P * 32, (size_t)(E - B) * 32, (size_t)n_c,
                         cudaMemcpyHostToDevice, c->copy_stream));
    CU(cudaMemcpyAsync(d_rf_all, ref + B, (size_t)(E - B), cudaMemcpyHostToDevice, c->copy_stream));
    CU(c->calls.need(sizeof(as_call) * (size_t)std::max<int64_t>(cap, 1) * (size_t)n_c));
    CU(c->misc.need(16 * 8));
    CU(c->h_small.need(8 * 8));
    // d_n[i] = calls of table i found so far, d_n[8 + i] = the count before the current tile
    unsigned long long* d_n = (unsigned long long*)c->misc.p;
    unsigned long long* h_total = (unsigned long long*)c->h_small.p;
    CU(cudaMemsetAsync(d_n, 0, 16 * 8, c->exec_stream));
    const bool sweep = n_c > 1;
    const bool deferred = sweep && (c->call_variant == AS_DEFERRED_CALL_KERNEL || c->call_variant == AS_DEFAULT_CALL_KERNEL);
    const int64_t ntiles = (E - B + TP - 1) / TP;
    clk.lap("call.checks_alloc");
    CU(stage_wide(c, src, c->copy_stream));
    clk.lap("call.stage_wide");
    int ret = AS_OK;
    for (int64_t t = 0; t < ntiles && ret == AS_OK; ++t) {
        const int bsel = (int)(t & 1);
        const int64_t p0 = B + t * TP, n = std::min(TP, E - p0);
#define CUB(call) { cudaError_t e_ = (call); if (e_ != cudaSuccess) { ret = fail(AS_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); break; } }
        if (t >= 2) CUB(cudaStreamWaitEvent(c->copy_stream, c->ev_done[bsel], 0));
        CUB(upload_tile(c, bsel, src, T, P, p0, n, c->copy_stream));
        CUB(cudaEventRecord(c->ev_up[bsel], c->copy_stream));
        CUB(cudaStreamWaitEvent(c->exec_stream, c->ev_up[bsel], 0));
        CUB(expand_tile(c, bsel, src, T, p0, n, c->exec_stream));
        // the tile kernel emits tile-local slot ids; the entries it appended, [d_n[8 + i], d_n[i]), get the tile offset
        if (p0 > 0) CUB(cudaMemcpyAsync(d_n + 8, d_n, 8 * (size_t)n_c, cudaMemcpyDeviceToDevice, c->exec_stream));
        const uint32_t* d_tile = (const uint32_t*)c->tile[bsel].p;
        if (deferred) {
            if ((ret = call_deferred(c, d_tile, T, n, 0, n, d_rf_all + (p0 - B), d_tv_all + (p0 - B) * 8, n_c, c_stride, cut,
                                     (as_call*)c->calls.p, cap, d_n, c->exec_stream)) != AS_OK)
                break;
        } else {
            CUB(as_launch_call_sweep(c->call_variant, d_tile, T, n, 0, n, d_rf_all + (p0 - B), d_tv_all + (p0 - B) * 8, n_c, c_stride,
                                     (uint32_t)cut, (as_call*)c->calls.p, cap, d_n, c->fwd_pending_cap, c->exec_stream));
            c->launches += 1;
        }
        if (p0 > 0) {
            for (int32_t i = 0; i < n_c; ++i) {
                CUB(as_launch_call_slot_offset((as_call*)c->calls.p + i * cap, d_n + 8 + i, d_n + i, cap, (int32_t)p0, c->exec_stream));
                c->launches += 1;
            }
            if (ret != AS_OK) break;
        }
        CUB(cudaEventRecord(c->ev_done[bsel], c->exec_stream));
#undef CUB
    }
    clk.lap("call.enqueue");
    if (ret == AS_OK) {
        cudaError_t e0 = cudaMemcpyAsync(h_total, d_n, 8 * (size_t)n_c, cudaMemcpyDeviceToHost, c->exec_stream);
        cudaError_t e1 = cudaStreamSynchronize(c->exec_stream), e2 = cudaStreamSynchronize(c->copy_stream);
        clk.lap("call.drain");
        if (e0 != cudaSuccess || e1 != cudaSuccess || e2 != cudaSuccess)
            ret = fail(AS_ECUDA, "caller pipeline failed: %s", cudaGetErrorString(e0 != cudaSuccess ? e0 : e1 != cudaSuccess ? e1 : e2));
    }
    if (ret == AS_OK)
        for (int32_t i = 0; i < n_c; ++i) found[i] = (int64_t)h_total[i];
    return ret;
}

// ---- sharding of the _host entry points over the devices of a multi-device context ------------------------------------
// Contiguous, near-equal slot ranges whose boundaries are multiples of 128 where possible and never split a twin group
// (the noise model reduces all slots of a position together, EE:1241-1245).  twin_head may be NULL.
static std::vector<int64_t> shard_bounds(int64_t P, int n, const int32_t* twin_next, const int32_t* twin_head) {
    std::vector<int32_t> reach;  // reach[i] = the last slot of any group that has a member <= i (prefix maximum)
    if (twin_head && twin_next) {
        std::vector<int32_t> last((size_t)P);
        for (int64_t i = 0; i < P; ++i) last[(size_t)i] = (int32_t)i;
        for (int64_t i = 0; i < P; ++i) {  // members are chained in ascending order: the last write per head is the maximum
            const int32_t h = twin_head[i];
            if (h >= 0 && h < P && last[(size_t)h] < (int32_t)i) last[(size_t)h] = (int32_t)i;
        }
        reach.resize((size_t)P);
        int32_t m = -1;
        for (int64_t i = 0; i < P; ++i) {
            const int32_t h = twin_head[i];
            if (h >= 0 && h < P) m = std::max(m, last[(size_t)h]);
            reach[(size_t)i] = m;
        }
    }
    std::vector<int64_t> bounds(1, 0);
    for (int r = 1; r < n; ++r) {
        int64_t b = (P * r / n) / 128 * 128;
        b = std::max(b, bounds.back());
        if (!reach.empty())
            while (b > 0 && b < P && reach[(size_t)b - 1] >= b) b = (int64_t)reach[(size_t)b - 1] + 1;  // a group that starts below b ends at or after b
        bounds.push_back(std::min(b, P));
    }
    bounds.push_back(P);
    return bounds;
}

// the same partition for callers that place the shards themselves (one process per GPU: bench.py, amplisolve_b200/shard.py)
int as_shard_bounds(int64_t P, int32_t n_shards, const int32_t* twin_next, const int32_t* twin_head, int64_t* bounds_out) {
    if (P < 0 || n_shards < 1 || !bounds_out) return fail(AS_EINVAL, "bad argument");
    if ((twin_next == nullptr) != (twin_head == nullptr)) return fail(AS_EINVAL, "twin_next and twin_head go together");
    const std::vector<int64_t> b = shard_bounds(P, n_shards, twin_next, twin_head);
    for (size_t i = 0; i < b.size(); ++i) bounds_out[i] = b[i];
    return AS_OK;
}

struct ShardResult {
    int rc = AS_OK;
    char err[512] = "";
    int64_t found = 0;
};

}  // extern "C"
template <class F>
static int run_on_devices(as_ctx* c, F body) {  // body(k, sub-context) on one host thread per device
    const int n = (int)c->subs.size();
    std::vector<ShardResult> res((size_t)n);
    auto work = [&](int k) {
        res[(size_t)k].rc = body(k, c->subs[(size_t)k], res[(size_t)k]);
        if (res[(size_t)k].rc != AS_OK) snprintf(res[(size_t)k].err, sizeof res[(size_t)k].err, "%s", g_err);
    };
    std::vector<std::thread> th;
    for (int k = 1; k < n; ++k) th.emplace_back(work, k);
    work(0);
    for (auto& t : th) t.join();
    cudaSetDevice(c->device);
    for (int k = 0; k < n; ++k)
        if (res[(size_t)k].rc != AS_OK) return fail(res[(size_t)k].rc, "device %d: %s", c->subs[(size_t)k]->device, res[(size_t)k].err);
    return AS_OK;
}
extern "C" {

static int noise_estimate_host_impl(as_ctx* c, const HostSrc& src, int32_t S, int64_t P, const int32_t* twin_next,
                                    const int32_t* twin_head, const float* c_values, int32_t n_c, int32_t cut, float* thr,
                                    float* germ_val, uint8_t* germ_state, uint32_t* count, uint32_t* nrec, float* thr_view) {
    if (!c_values || n_c < 1 || n_c > 8) return fail(AS_EINVAL, "a sweep takes 1..8 values of C");
    int rc = check_common(c, src.counts, S, P, 0, P, cut);
    if (rc) return rc;
    if ((rc = check_wide(src, S, P)) != AS_OK) return rc;
    if (!thr || !germ_val || !germ_state || !count || !nrec) return fail(AS_EINVAL, "output pointer is NULL");
    if ((twin_next == nullptr) != (twin_head == nullptr)) return fail(AS_EINVAL, "twin_next and twin_head go together");
    if (P == 0) return AS_OK;
    if (c->subs.size() < 2)
        return noise_estimate_host_range(c, src, S, P, 0, P, twin_next, twin_head, c_values, n_c, cut, thr, germ_val, germ_state, count,
                                         nrec, thr_view);
    const std::vector<int64_t> bounds = shard_bounds(P, (int)c->subs.size(), twin_next, twin_head);
    return run_on_devices(c, [&](int k, as_ctx* sub, ShardResult&) {
        return noise_estimate_host_range(sub, src, S, P, bounds[(size_t)k], bounds[(size_t)k + 1], twin_next, twin_head, c_values, n_c,
                                         cut, thr, germ_val, germ_state, count, nrec, thr_view);
    });
}

// n_c tables: calls [n_c][cap], n_calls [n_c].  Each table's lists of all devices meet on the first one (peer copies of
// exact sizes), are sorted there into the reference's row order (sample, slot, alt), one radix sort per table, and come
// down with one copy per table.
static int call_variants_host_impl(as_ctx* c, const HostSrc& src, int32_t T, int64_t P, const uint8_t* ref,
                                   const float* thr_views, int32_t n_c, int32_t cut, as_call* calls, int64_t cap, int64_t* n_calls) {
    PhaseClock clk;
    if (n_c < 1 || n_c > 8) return fail(AS_EINVAL, "a sweep takes 1..8 threshold tables");
    int rc = check_common(c, src.counts, T, P, 0, P, cut);
    if (rc) return rc;
    if ((rc = check_wide(src, T, P)) != AS_OK) return rc;
    if (!ref || !thr_views || !n_calls || (!calls && cap > 0) || cap < 0) return fail(AS_EINVAL, "bad pointer / cap");
    if (c->call_variant < 2 && n_c > 1) return fail(AS_EINVAL, "the sweep needs a TMA-staged caller variant (>= 2)");
    for (int32_t i = 0; i < n_c; ++i) n_calls[i] = 0;
    if (P == 0 || T == 0) return AS_OK;
    const int ndev = c->subs.size() < 2 ? 1 : (int)c->subs.size();
    std::vector<int64_t> found((size_t)ndev * 8, 0);  // found[k * 8 + i]: device k, table i
    if (ndev == 1) {
        rc = call_variants_host_range(c, src, T, P, 0, P, ref, thr_views, n_c, cut, cap, &found[0]);
    } else {
        const std::vector<int64_t> bounds = shard_bounds(P, ndev, nullptr, nullptr);
        rc = run_on_devices(c, [&](int k, as_ctx* sub, ShardResult&) {
            return call_variants_host_range(sub, src, T, P, bounds[(size_t)k], bounds[(size_t)k + 1], ref, thr_views, n_c, cut, cap,
                                            &found[(size_t)k * 8]);
        });
    }
    if (rc != AS_OK) return rc;
    CU(cudaSetDevice(c->device));
    std::vector<int64_t> have((size_t)n_c, 0);
    int64_t max_have = 0, sum_list = 0;
    bool over = false;
    for (int32_t i = 0; i < n_c; ++i) {
        int64_t total = 0;
        for (int k = 0; k < ndev; ++k) {
            const int64_t f = found[(size_t)k * 8 + i];
            total += f;
            have[(size_t)i] += std::min(f, cap);
            over = over || f > cap;
        }
        n_calls[i] = total;
        over = over || total > cap;
        max_have = std::max(max_have, have[(size_t)i]);
        sum_list += (int64_t)(((size_t)have[(size_t)i] * sizeof(as_call) + 255) & ~(size_t)255);
    }
    if (max_have > 0) {
        // sortbuf: sorted lists of every table | sort scratch | gathered list of one table (several devices)
        const size_t scratch = as_sort_calls_scratch_bytes(max_have);
        const size_t gather = ndev > 1 ? (size_t)max_have * sizeof(as_call) : 0;
        CU(c->sortbuf.need((size_t)sum_list + scratch + gather));
        char* sorted = (char*)c->sortbuf.p;
        char* sort_scratch = sorted + sum_list;
        for (int32_t i = 0; i < n_c; ++i) {
            const int64_t h = have[(size_t)i];
            if (h == 0) continue;
            as_call* gathered = (as_call*)c->calls.p + i * cap;
            if (ndev > 1) {
                gathered = (as_call*)(sort_scratch + scratch);
                int64_t off = 0;
                for (int k = 0; k < ndev; ++k) {
                    const int64_t n = std::min(found[(size_t)k * 8 + i], cap);
                    if (n > 0) CU(cudaMemcpyPeerAsync(gathered + off, c->device, (as_call*)c->subs[(size_t)k]->calls.p + i * cap,
                                                      c->subs[(size_t)k]->device, sizeof(as_call) * (size_t)n, c->exec_stream));
                    off += n;
                }
            }
            CU(as_launch_sort_calls(gathered, h, (as_call*)sorted, sort_scratch, scratch, c->exec_stream));
            c->launches += 3;
            CU(cudaMemcpyAsync(calls + i * cap, sorted, sizeof(as_call) * (size_t)std::min(h, cap), cudaMemcpyDeviceToHost,
                               c->exec_stream));
            sorted += ((size_t)h * sizeof(as_call) + 255) & ~(size_t)255;
        }
        CU(cudaStreamSynchronize(c->exec_stream));
        clk.lap("call.sort_download");
    }
    if (over) {
        int32_t worst = 0;
        for (int32_t i = 1; i < n_c; ++i) if (n_calls[i] > n_calls[worst]) worst = i;
        return fail(AS_EOVERFLOW, "%lld calls found, capacity %lld", (long long)n_calls[worst], (long long)cap);
    }
    return AS_OK;
}

int as_noise_estimate_host(as_ctx* c, const uint32_t* counts, int32_t S, int64_t P, const int32_t* twin_next,
                           const int32_t* twin_head, float C, int32_t cut, float* thr, float* germ_val,
                           uint8_t* germ_state, uint32_t* count, uint32_t* nrec, float* thr_view) {
    const HostSrc src{counts, 4, nullptr, 0};
    return noise_estimate_host_impl(c, src, S, P, twin_next, twin_head, &C, 1, cut, thr, germ_val, germ_state, count, nrec, thr_view);
}
int as_noise_estimate_host16(as_ctx* c, const uint16_t* counts, const as_wide_record* wide, int64_t n_wide, int32_t S,
                             int64_t P, const int32_t* twin_next, const int32_t* twin_head, float C, int32_t cut, float* thr,
                             float* germ_val, uint8_t* germ_state, uint32_t* count, uint32_t* nrec, float* thr_view) {
    const HostSrc src{counts, 2, wide, n_wide};
    return noise_estimate_host_impl(c, src, S, P, twin_next, twin_head, &C, 1, cut, thr, germ_val, germ_state, count, nrec, thr_view);
}
int as_call_variants_host(as_ctx* c, const uint32_t* counts, int32_t T, int64_t P, const uint8_t* ref,
                          const float* thr_view, int32_t cut, as_call* calls, int64_t cap, int64_t* n_calls) {
    const HostSrc src{counts, 4, nullptr, 0};
    return call_variants_host_impl(c, src, T, P, ref, thr_view, 1, cut, calls, cap, n_calls);
}
int as_noise_estimate_host_packed(as_ctx* c, const uint32_t* packed, const as_wide_record* wide, int64_t n_wide, int32_t S,
                                  int64_t P, const int32_t* twin_next, const int32_t* twin_head, float C, int32_t cut,
                                  float* thr, float* germ_val, uint8_t* germ_state, uint32_t* count, uint32_t* nrec,
                                  float* thr_view) {
    const HostSrc src{packed, 1, wide, n_wide};
    return noise_estimate_host_impl(c, src, S, P, twin_next, twin_head, &C, 1, cut, thr, germ_val, germ_state, count, nrec, thr_view);
}
int as_call_variants_host_packed(as_ctx* c, const uint32_t* packed, const as_wide_record* wide, int64_t n_wide, int32_t T,
                                 int64_t P, const uint8_t* ref, const float* thr_view, int32_t cut, as_call* calls,
                                 int64_t cap, int64_t* n_calls) {
    const HostSrc src{packed, 1, wide, n_wide};
    return call_variants_host_impl(c, src, T, P, ref, thr_view, 1, cut, calls, cap, n_calls);
}

// uint32 counts -> packed wire format + escaped records.  Threads over samples; the per-sample lists are concatenated
// and sorted by (slot, sample).
int as_pack_counts(const uint32_t* counts, int32_t n_samples, int64_t P, uint32_t* packed, as_wide_record* wide,
                   int64_t wide_cap, int64_t* n_wide) {
    if (!counts || !packed || !n_wide || n_samples < 0 || P < 0 || wide_cap < 0 || (wide_cap > 0 && !wide))
        return fail(AS_EINVAL, "bad argument");
    *n_wide = 0;
    std::vector<std::vector<as_wide_record>> per((size_t)n_samples);
    std::atomic<int32_t> next(0);
    auto work = [&]() {
        for (int32_t s = next.fetch_add(1); s < n_samples; s = next.fetch_add(1)) {
            const uint32_t* f = counts + ((int64_t)s * 2) * P * 4;
            const uint32_t* b = f + P * 4;
            uint32_t* pf = packed + ((int64_t)s * 2) * P;
            uint32_t* pb = pf + P;
            for (int64_t p = 0; p < P; ++p) {
                if (f[p * 4] == AS_ABSENT) { pf[p] = pb[p] = AS_PACKED_ABSENT; continue; }
                uint32_t wf, wb;
                if (as_pack_word(f + p * 4, &wf) && as_pack_word(b + p * 4, &wb)) { pf[p] = wf; pb[p] = wb; continue; }
                pf[p] = pb[p] = AS_PACKED_ESCAPE;
                as_wide_record r;
                r.sample = s;
                r.slot = (int32_t)p;
                memcpy(r.fw, f + p * 4, 16);
                memcpy(r.bw, b + p * 4, 16);
                per[(size_t)s].push_back(r);
            }
        }
    };
    const unsigned hw = std::max(1u, std::min(std::thread::hardware_concurrency(), (unsigned)std::max(1, n_samples)));
    std::vector<std::thread> th;
    for (unsigned t = 1; t < hw; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
    int64_t total = 0;
    for (const auto& v : per) total += (int64_t)v.size();
    *n_wide = total;
    if (total > wide_cap) return fail(AS_EOVERFLOW, "%lld records escape the packed format, capacity %lld", (long long)total, (long long)wide_cap);
    int64_t k = 0;
    for (const auto& v : per) { if (!v.empty()) memcpy(wide + k, v.data(), v.size() * sizeof(as_wide_record)); k += (int64_t)v.size(); }
    std::sort(wide, wide + total, [](const as_wide_record& x, const as_wide_record& y) {
        return x.slot != y.slot ? x.slot < y.slot : x.sample < y.sample;
    });
    return AS_OK;
}

int as_call_variants_host16(as_ctx* c, const uint16_t* counts, const as_wide_record* wide, int64_t n_wide, int32_t T,
                            int64_t P, const uint8_t* ref, const float* thr_view, int32_t cut, as_call* calls, int64_t cap,
                            int64_t* n_calls) {
    const HostSrc src{counts, 2, wide, n_wide};
    return call_variants_host_impl(c, src, T, P, ref, thr_view, 1, cut, calls, cap, n_calls);
}

// Noise-floor sweep on the _host path: n_c values of C / n_c threshold tables through the same pipelines
int as_noise_estimate_sweep_host(as_ctx* c, const uint32_t* counts, int32_t S, int64_t P, const int32_t* twin_next,
                                 const int32_t* twin_head, const float* c_values, int32_t n_c, int32_t cut, float* thr,
                                 float* germ_val, uint8_t* germ_state, uint32_t* count, uint32_t* nrec, float* thr_view) {
    const HostSrc src{counts, 4, nullptr, 0};
    return noise_estimate_host_impl(c, src, S, P, twin_next, twin_head, c_values, n_c, cut, thr, germ_val, germ_state, count, nrec,
                                    thr_view);
}
int as_noise_estimate_sweep_host16(as_ctx* c, const uint16_t* counts, const as_wide_record* wide, int64_t n_wide, int32_t S,
                                   int64_t P, const int32_t* twin_next, const int32_t* twin_head, const float* c_values,
                                   int32_t n_c, int32_t cut, float* thr, float* germ_val, uint8_t* germ_state, uint32_t* count,
                                   uint32_t* nrec, float* thr_view) {
    const HostSrc src{counts, 2, wide, n_wide};
    return noise_estimate_host_impl(c, src, S, P, twin_next, twin_head, c_values, n_c, cut, thr, germ_val, germ_state, count, nrec,
                                    thr_view);
}
int as_noise_estimate_sweep_host_packed(as_ctx* c, const uint32_t* packed, const as_wide_record* wide, int64_t n_wide, int32_t S,
                                        int64_t P, const int32_t* twin_next, const int32_t* twin_head, const float* c_values,
                                        int32_t n_c, int32_t cut, float* thr, float* germ_val, uint8_t* germ_state,
                                        uint32_t* count, uint32_t* nrec, float* thr_view) {
    const HostSrc src{packed, 1, wide, n_wide};
    return noise_estimate_host_impl(c, src, S, P, twin_next, twin_head, c_values, n_c, cut, thr, germ_val, germ_state, count, nrec,
                                    thr_view);
}
int as_call_variants_sweep_host(as_ctx* c, const uint32_t* counts, int32_t T, int64_t P, const uint8_t* ref,
                                const float* thr_views, int32_t n_c, int32_t cut, as_call* calls, int64_t cap, int64_t* n_calls) {
    const HostSrc src{counts, 4, nullptr, 0};
    return call_variants_host_impl(c, src, T, P, ref, thr_views, n_c, cut, calls, cap, n_calls);
}
int as_call_variants_sweep_host16(as_ctx* c, const uint16_t* counts, const as_wide_record* wide, int64_t n_wide, int32_t T,
                                  int64_t P, const uint8_t* ref, const float* thr_views, int32_t n_c, int32_t cut, as_call* calls,
                                  int64_t cap, int64_t* n_calls) {
    const HostSrc src{counts, 2, wide, n_wide};
    return call_variants_host_impl(c, src, T, P, ref, thr_views, n_c, cut, calls, cap, n_calls);
}
int as_call_variants_sweep_host_packed(as_ctx* c, const uint32_t* packed, const as_wide_record* wide, int64_t n_wide, int32_t T,
                                       int64_t P, const uint8_t* ref, const float* thr_views, int32_t n_c, int32_t cut,
                                       as_call* calls, int64_t cap, int64_t* n_calls) {
    const HostSrc src{packed, 1, wide, n_wide};
    return call_variants_host_impl(c, src, T, P, ref, thr_views, n_c, cut, calls, cap, n_calls);
}

// ---- site report ---------------------------------------------------------------------------------------------------
// The sites' columns of the host tensor are gathered in its own format into pinned memory ([T][2][H] words), go up as a count
// tensor of H slots and through the path of an upload tile (widen / unpack, escaped records patched in after renumbering them
// by site); site_test_kernel then evaluates every (table, site, tumour, strand) into out [n_c][T][H].
static int site_tests_impl(as_ctx* c, const HostSrc& src, int32_t T, int64_t P, const uint8_t* ref, const float* thr_views,
                           int32_t n_c, const int32_t* site_slot, const int32_t* site_alt, int64_t H, int32_t cut, as_site_test* out) {
    if (n_c < 1 || n_c > 8) return fail(AS_EINVAL, "site tests take 1..8 threshold tables");
    int rc = check_common(c, src.counts, T, P, 0, P, cut);
    if (rc) return rc;
    if (H < 0 || H > 0x7fffffffll) return fail(AS_EINVAL, "bad number of sites %lld", (long long)H);
    if (H > 0 && (!ref || !thr_views || !site_slot || !site_alt || !out)) return fail(AS_EINVAL, "bad pointer");
    for (int64_t h = 0; h < H; ++h) {
        if (site_slot[h] < 0 || site_slot[h] >= P)
            return fail(AS_EINVAL, "site %lld: slot %d outside [0, %lld)", (long long)h, site_slot[h], (long long)P);
        if (site_alt[h] < 0 || site_alt[h] > 3) return fail(AS_EINVAL, "site %lld: alt %d is not 0..3", (long long)h, site_alt[h]);
    }
    if (H == 0 || T == 0) return AS_OK;
    if ((rc = check_wide(src, T, P)) != AS_OK) return rc;
    PhaseClock clk;
    CU(cudaSetDevice(c->device));
    const size_t word = (size_t)src.elem * 4;  // bytes per (sample, strand, slot) in the host format
    const int64_t rows = (int64_t)T * 2;
    const size_t n_words = (size_t)rows * (size_t)H;
    std::vector<as_wide_record> wide;  // escaped records of the sites' slots, slot = site index
    if (src.elem != 4)
        for (int64_t h = 0; h < H; ++h) {
            const as_wide_record* r = std::lower_bound(src.wide, src.wide + src.n_wide, (int64_t)site_slot[h],
                                                       [](const as_wide_record& x, int64_t v) { return (int64_t)x.slot < v; });
            for (; r < src.wide + src.n_wide && r->slot == site_slot[h]; ++r) {
                wide.push_back(*r);
                wide.back().slot = (int32_t)h;
            }
        }
    // pinned host block: gathered columns | site_ra [H] | thr [n_c][H][2]
    const size_t o_ra = (n_words * word + 15) & ~(size_t)15;
    const size_t o_thr = (o_ra + (size_t)H * 2 + 15) & ~(size_t)15;
    const size_t h_bytes = o_thr + (size_t)n_c * (size_t)H * 8;
    CU(c->h_sites.need(h_bytes));
    char* hb = (char*)c->h_sites.p;
    {
        const int nth = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(std::thread::hardware_concurrency(), 16u), rows / 64));
        auto work = [&](int k) {
            for (int64_t r = rows * k / nth; r < rows * (k + 1) / nth; ++r) {
                const char* row = (const char*)src.counts + (size_t)r * (size_t)P * word;
                char* dst = hb + (size_t)r * (size_t)H * word;
                for (int64_t h = 0; h < H; ++h) memcpy(dst + (size_t)h * word, row + (size_t)site_slot[h] * word, word);
            }
        };
        std::vector<std::thread> th;
        for (int k = 1; k < nth; ++k) th.emplace_back(work, k);
        work(0);
        for (auto& x : th) x.join();
    }
    uint16_t* ra = (uint16_t*)(hb + o_ra);
    float* thr = (float*)(hb + o_thr);
    for (int64_t h = 0; h < H; ++h) {
        const int64_t s = site_slot[h], a = site_alt[h];
        ra[h] = (uint16_t)(ref[s] | (a << 8));
        for (int32_t i = 0; i < n_c; ++i) {
            thr[((int64_t)i * H + h) * 2 + 0] = thr_views[(((int64_t)i * P + s) * 4 + a) * 2 + 0];
            thr[((int64_t)i * H + h) * 2 + 1] = thr_views[(((int64_t)i * P + s) * 4 + a) * 2 + 1];
        }
    }
    clk.lap("sites.gather");
    // device block: tile [T][2][H][4] | staging (wire formats) | wide | site_ra | thr | out
    const size_t d_stg = n_words * 16;
    const size_t d_wide = d_stg + (src.elem == 4 ? 0 : ((n_words * word + 15) & ~(size_t)15));
    const size_t d_ra = d_wide + wide.size() * sizeof(as_wide_record);
    const size_t d_out = (d_ra + (h_bytes - o_ra) + 15) & ~(size_t)15;
    const size_t out_bytes = (size_t)n_c * (size_t)T * (size_t)H * sizeof(as_site_test);
    CU(c->sites.need(d_out + out_bytes));
    char* db = (char*)c->sites.p;
    cudaStream_t st = c->exec_stream;
    cudaEvent_t ev[5] = {};
    if (clk.on)
        for (cudaEvent_t& x : ev) CU(cudaEventCreate(&x));
    if (clk.on) CU(cudaEventRecord(ev[0], st));
    CU(cudaMemcpyAsync(db + (src.elem == 4 ? 0 : d_stg), hb, n_words * word, cudaMemcpyHostToDevice, st));
    if (!wide.empty())
        CU(cudaMemcpyAsync(db + d_wide, wide.data(), wide.size() * sizeof(as_wide_record), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(db + d_ra, hb + o_ra, h_bytes - o_ra, cudaMemcpyHostToDevice, st));
    if (clk.on) CU(cudaEventRecord(ev[1], st));
    if (src.elem != 4) {
        CU(src.elem == 2 ? as_launch_widen16((const uint16_t*)(db + d_stg), (uint32_t*)db, (int64_t)n_words, st)
                         : as_launch_unpack((const uint32_t*)(db + d_stg), (uint32_t*)db, (int64_t)n_words, st));
        c->launches += 1;
        if (!wide.empty()) {
            CU(as_launch_patch_wide((const as_wide_record*)(db + d_wide), (int64_t)wide.size(), (uint32_t*)db, H, 0, T, st));
            c->launches += 1;
        }
    }
    if (clk.on) CU(cudaEventRecord(ev[2], st));
    CU(as_launch_site_test((const uint32_t*)db, T, (int)H, (const uint16_t*)(db + d_ra), (const float*)(db + d_ra + (o_thr - o_ra)), n_c,
                           (uint32_t)cut, (as_site_test*)(db + d_out), st));
    c->launches += 1;
    if (clk.on) CU(cudaEventRecord(ev[3], st));
    CU(cudaMemcpyAsync(out, db + d_out, out_bytes, cudaMemcpyDeviceToHost, st));
    if (clk.on) CU(cudaEventRecord(ev[4], st));
    CU(cudaStreamSynchronize(st));
    if (clk.on) {
        const char* name[4] = {"upload", "expand", "kernel", "download"};
        for (int i = 0; i < 4; ++i) {
            float ms = 0.f;
            CU(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
            fprintf(stderr, "AS_TIMING capi.sites.%s_event %.6f\n", name[i], ms * 1e-3);
        }
        for (cudaEvent_t x : ev) cudaEventDestroy(x);
    }
    clk.lap("sites.device");
    return AS_OK;
}

int as_site_tests_host(as_ctx* c, const uint32_t* counts, int32_t T, int64_t P, const uint8_t* ref, const float* thr_views,
                       int32_t n_c, const int32_t* site_slot, const int32_t* site_alt, int64_t n_sites, int32_t cut, as_site_test* out) {
    const HostSrc src{counts, 4, nullptr, 0};
    return site_tests_impl(c, src, T, P, ref, thr_views, n_c, site_slot, site_alt, n_sites, cut, out);
}
int as_site_tests_host16(as_ctx* c, const uint16_t* counts, const as_wide_record* wide, int64_t n_wide, int32_t T, int64_t P,
                         const uint8_t* ref, const float* thr_views, int32_t n_c, const int32_t* site_slot, const int32_t* site_alt,
                         int64_t n_sites, int32_t cut, as_site_test* out) {
    const HostSrc src{counts, 2, wide, n_wide};
    return site_tests_impl(c, src, T, P, ref, thr_views, n_c, site_slot, site_alt, n_sites, cut, out);
}
int as_site_tests_host_packed(as_ctx* c, const uint32_t* packed, const as_wide_record* wide, int64_t n_wide, int32_t T, int64_t P,
                              const uint8_t* ref, const float* thr_views, int32_t n_c, const int32_t* site_slot,
                              const int32_t* site_alt, int64_t n_sites, int32_t cut, as_site_test* out) {
    const HostSrc src{packed, 1, wide, n_wide};
    return site_tests_impl(c, src, T, P, ref, thr_views, n_c, site_slot, site_alt, n_sites, cut, out);
}

// Device call list -> the reference's row order (sample, slot, alt), on the device (radix sort of 64-bit keys + row gather).
// slot_offset is added to every slot first (a shard's local slot ids -> panel slot ids).
int as_sort_calls_dev(as_ctx* c, as_call* d_calls, int64_t n, int32_t slot_offset, as_call* d_sorted, void* stream) {
    if (!c || n < 0 || (n > 0 && (!d_calls || !d_sorted))) return fail(AS_EINVAL, "bad argument");
    if (n == 0) return AS_OK;
    if (n > 0x7fffffffll) return fail(AS_EINVAL, "at most 2^31-1 calls per sort");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t scratch = as_sort_calls_scratch_bytes(n);
    CU(c->sortbuf.need(scratch + 64));
    CU(c->misc.need(32));
    if (slot_offset != 0) {
        unsigned long long h[2] = {0ull, (unsigned long long)n};
        CU(cudaMemcpyAsync(c->misc.p, h, 16, cudaMemcpyHostToDevice, st));
        CU(as_launch_call_slot_offset(d_calls, (const unsigned long long*)c->misc.p, (const unsigned long long*)c->misc.p + 1, n,
                                      slot_offset, st));
        c->launches += 1;
    }
    CU(as_launch_sort_calls(d_calls, n, d_sorted, c->sortbuf.p, scratch, st));
    c->launches += 3;
    return AS_OK;
}

// ---- pileup (SURVEY.md 8 f4): BAM records -> counts[2][P][4] of one sample -----------------------------
int as_pileup_begin(as_ctx* c, const int64_t* contig_first, int32_t n_contig, const int32_t* slot_pos, int64_t P) {
    if (!c || !contig_first || !slot_pos || n_contig < 1 || P < 1) return fail(AS_EINVAL, "bad argument");
    if (contig_first[0] != 0 || contig_first[n_contig] != P) return fail(AS_EINVAL, "contig_first must run from 0 to P");
    for (int32_t k = 0; k < n_contig; ++k) {
        if (contig_first[k + 1] < contig_first[k]) return fail(AS_EINVAL, "contig_first must not decrease");
        for (int64_t j = contig_first[k] + 1; j < contig_first[k + 1]; ++j)
            if (slot_pos[j] <= slot_pos[j - 1]) return fail(AS_EINVAL, "positions of contig %d are not sorted and unique", k);
    }
    if (c->subs.size() > 1) c = c->subs[0];  // one sample, one GPU
    CU(cudaSetDevice(c->device));
    CU(c->pile_first.need(sizeof(int64_t) * (size_t)(n_contig + 1)));
    CU(c->pile_pos.need(sizeof(int32_t) * (size_t)P));
    CU(c->pile_counts.need(sizeof(uint32_t) * 8 * (size_t)P));
    CU(c->pile_stats.need(16));
    cudaStream_t st = c->exec_stream;
    CU(cudaMemcpyAsync(c->pile_first.p, contig_first, sizeof(int64_t) * (size_t)(n_contig + 1), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(c->pile_pos.p, slot_pos, sizeof(int32_t) * (size_t)P, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(c->pile_counts.p, 0, sizeof(uint32_t) * 8 * (size_t)P, st));
    CU(cudaMemsetAsync(c->pile_stats.p, 0, 16, st));
    CU(cudaStreamSynchronize(st));  // the host arrays may go away
    c->pile_P = P;
    c->pile_contigs = n_contig;
    return AS_OK;
}

int as_pileup_add_host(as_ctx* c, const uint8_t* records, int64_t n_bytes, const int64_t* rec_off, int64_t n_rec,
                       const int32_t* ref_contig, int32_t n_ref, int32_t mbq, int32_t mrq, uint32_t skip_flags) {
    if (!c || n_bytes < 0 || n_rec < 0 || n_ref < 1 || !ref_contig) return fail(AS_EINVAL, "bad argument");
    if (c->subs.size() > 1) c = c->subs[0];
    if (c->pile_P < 1) return fail(AS_EINVAL, "as_pileup_begin has not been called");
    if (n_rec == 0) return AS_OK;
    if (!records || !rec_off) return fail(AS_EINVAL, "records / rec_off is NULL");
    for (int32_t k = 0; k < n_ref; ++k)
        if (ref_contig[k] < -1 || ref_contig[k] >= c->pile_contigs) return fail(AS_EINVAL, "ref_contig[%d] names no panel contig", k);
    for (int64_t i = 0; i < n_rec; ++i)
        if (rec_off[i] < 0 || rec_off[i] + 36 > n_bytes) return fail(AS_EINVAL, "record %lld starts outside the buffer", (long long)i);
    CU(cudaSetDevice(c->device));
    CU(c->pile_rec.need((size_t)n_bytes + 16));
    CU(c->pile_off.need(sizeof(int64_t) * (size_t)n_rec));
    CU(c->pile_ref.need(sizeof(int32_t) * (size_t)n_ref));
    cudaStream_t st = c->exec_stream;
    const bool timing = getenv("AS_TIMING") != nullptr;
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    if (timing) {
        for (auto& e : ev) CU(cudaEventCreate(&e));
        CU(cudaEventRecord(ev[0], st));
    }
    CU(cudaMemcpyAsync(c->pile_rec.p, records, (size_t)n_bytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(c->pile_off.p, rec_off, sizeof(int64_t) * (size_t)n_rec, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(c->pile_ref.p, ref_contig, sizeof(int32_t) * (size_t)n_ref, cudaMemcpyHostToDevice, st));
    if (timing) CU(cudaEventRecord(ev[1], st));
    CU(as_launch_pileup((const uint8_t*)c->pile_rec.p, (const int64_t*)c->pile_off.p, n_rec, n_bytes, (const int32_t*)c->pile_ref.p, n_ref,
                        (const int64_t*)c->pile_first.p, (const int32_t*)c->pile_pos.p, c->pile_P, mbq, mrq, skip_flags,
                        (uint32_t*)c->pile_counts.p, (unsigned long long*)c->pile_stats.p, st));
    c->launches += 1;
    if (timing) CU(cudaEventRecord(ev[2], st));
    CU(cudaStreamSynchronize(st));  // the caller reuses its buffers for the next piece
    if (timing) {
        float a = 0, b = 0;
        CU(cudaEventElapsedTime(&a, ev[0], ev[1]));
        CU(cudaEventElapsedTime(&b, ev[1], ev[2]));
        c->pile_h2d_ms += a;
        c->pile_kernel_ms += b;
        for (auto& e : ev) cudaEventDestroy(e);
    }
    return AS_OK;
}

int as_pileup_end_host(as_ctx* c, uint32_t* counts, uint64_t* stats_out) {
    if (!c || !counts) return fail(AS_EINVAL, "bad argument");
    if (c->subs.size() > 1) c = c->subs[0];
    if (c->pile_P < 1) return fail(AS_EINVAL, "as_pileup_begin has not been called");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->exec_stream;
    CU(cudaMemcpyAsync(counts, c->pile_counts.p, sizeof(uint32_t) * 8 * (size_t)c->pile_P, cudaMemcpyDeviceToHost, st));
    unsigned long long h[2] = {0ull, 0ull};
    CU(cudaMemcpyAsync(h, c->pile_stats.p, 16, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (stats_out) { stats_out[0] = h[0]; stats_out[1] = h[1]; }
    if (getenv("AS_TIMING")) {
        fprintf(stderr, "AS_TIMING capi.pileup.h2d %.6f\nAS_TIMING capi.pileup.kernel %.6f\n", 1e-3 * c->pile_h2d_ms, 1e-3 * c->pile_kernel_ms);
        c->pile_h2d_ms = c->pile_kernel_ms = 0;
    }
    c->pile_P = -1;
    return AS_OK;
}

int as_pileup_set_host(as_ctx* c, const uint32_t* counts) {
    if (!c || !counts) return fail(AS_EINVAL, "bad argument");
    if (c->subs.size() > 1) c = c->subs[0];
    if (c->pile_P < 1) return fail(AS_EINVAL, "as_pileup_begin has not been called");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->exec_stream;
    CU(cudaMemcpyAsync(c->pile_counts.p, counts, sizeof(uint32_t) * 8 * (size_t)c->pile_P, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    return AS_OK;
}

// The pileup of one sample -> its slice of a host wire tensor (pileup_encode_kernel), the escaped records sorted by slot.
int as_pileup_end_wire(as_ctx* c, const int32_t* slot_unique, int64_t P, int32_t mdc, int32_t fmt, int32_t sample, void* wire,
                       as_wide_record* wide, int64_t wide_cap, int64_t* n_wide, int64_t* rows_out, uint64_t* stats_out) {
    if (!c || !slot_unique || !wire || !n_wide || P < 1 || P > 0x7fffffffll || (fmt != 1 && fmt != 2) || wide_cap < 0 ||
        (wide_cap > 0 && !wide))
        return fail(AS_EINVAL, "bad argument");
    if (c->subs.size() > 1) c = c->subs[0];
    const int64_t U = c->pile_P;
    if (U < 1) return fail(AS_EINVAL, "as_pileup_begin has not been called");
    for (int64_t s = 0; s < P; ++s)
        if (slot_unique[s] < 0 || slot_unique[s] >= U)
            return fail(AS_EINVAL, "slot_unique[%lld] = %d is not a position of the pileup (0..%lld)", (long long)s, slot_unique[s], (long long)U - 1);
    CU(cudaSetDevice(c->device));
    const size_t wire_bytes = (size_t)P * 2 * (fmt == 1 ? 4 : 8);
    const int64_t keep = std::min<int64_t>(wide_cap, P);  // no more than P records can escape
    CU(c->pile_slots.need(sizeof(int32_t) * (size_t)P));
    CU(c->pile_wire.need(wire_bytes));
    CU(c->pile_wide.need(sizeof(as_wide_record) * (size_t)std::max<int64_t>(1, keep)));
    CU(c->misc.need(32));
    cudaStream_t st = c->exec_stream;
    const bool timing = getenv("AS_TIMING") != nullptr;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    if (timing) for (auto& e : ev) CU(cudaEventCreate(&e));
    CU(cudaMemcpyAsync(c->pile_slots.p, slot_unique, sizeof(int32_t) * (size_t)P, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(c->misc.p, 0, 16, st));
    if (timing) CU(cudaEventRecord(ev[0], st));
    CU(as_launch_pileup_encode(fmt, (const uint32_t*)c->pile_counts.p, U, (const int32_t*)c->pile_slots.p, P, mdc, sample, c->pile_wire.p,
                               (as_wide_record*)c->pile_wide.p, keep, (unsigned long long*)c->misc.p, st));
    c->launches += 1;
    if (timing) CU(cudaEventRecord(ev[1], st));
    unsigned long long h[4] = {0ull, 0ull, 0ull, 0ull};  // escaped, present; reads used, bases counted
    CU(cudaMemcpyAsync(wire, c->pile_wire.p, wire_bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h, c->misc.p, 16, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h + 2, c->pile_stats.p, 16, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const int64_t n = (int64_t)h[0];
    if (n > 0 && n <= keep) {
        CU(cudaMemcpyAsync(wide, c->pile_wide.p, sizeof(as_wide_record) * (size_t)n, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        std::sort(wide, wide + n, [](const as_wide_record& x, const as_wide_record& y) { return x.slot < y.slot; });
    }
    if (timing) {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, ev[0], ev[1]));
        for (auto& e : ev) cudaEventDestroy(e);
        fprintf(stderr, "AS_TIMING capi.pileup.h2d %.6f\nAS_TIMING capi.pileup.kernel %.6f\nAS_TIMING capi.pileup.encode %.6f\n",
                1e-3 * c->pile_h2d_ms, 1e-3 * c->pile_kernel_ms, 1e-3 * ms);
        c->pile_h2d_ms = c->pile_kernel_ms = 0;
    }
    *n_wide = n;
    if (rows_out) *rows_out = (int64_t)h[1];
    if (stats_out) { stats_out[0] = h[2]; stats_out[1] = h[3]; }
    if (n > wide_cap) return fail(AS_EOVERFLOW, "%lld records escape the wire format, capacity %lld", (long long)n, (long long)wide_cap);
    c->pile_P = -1;
    return AS_OK;
}

// ---- element-wise evaluators -----------------------------------------------------------------------
int as_poisson_test_host(as_ctx* c, const int32_t* k, const int32_t* rd, const float* err, int64_t n, double* p,
                         double* q) {
    if (!c || !k || !rd || !err || !p || !q || n < 0) return fail(AS_EINVAL, "bad argument");
    if (n == 0) return AS_OK;
    CU(cudaSetDevice(c->device));
    CU(c->misc.need((size_t)n * 28 + 64));
    char* base = (char*)c->misc.p;
    double* d_p = (double*)base;
    double* d_q = d_p + n;
    int32_t* d_k = (int32_t*)(d_q + n);
    int32_t* d_rd = d_k + n;
    float* d_err = (float*)(d_rd + n);
    cudaStream_t st = c->exec_stream;
    CU(cudaMemcpyAsync(d_k, k, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_rd, rd, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_err, err, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CU(as_launch_poisson_test(d_k, d_rd, d_err, n, d_p, d_q, st));
    c->launches += 1;
    CU(cudaMemcpyAsync(p, d_p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(q, d_q, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return AS_OK;
}

// Fisher strand-bias tests of n calls (VC:902, VC:3797-3814) on the device; see include/amplisolve_b200.h
extern "C" double as_fisher_test(int32_t fw, int32_t bw, int32_t alt_fw, int32_t alt_bw);  // as_host.cpp
int as_fisher_tests_host(as_ctx* c, const int32_t* tables, int64_t n, double* p) {
    if (!c || n < 0 || (n > 0 && (!tables || !p))) return fail(AS_EINVAL, "bad argument");
    if (n == 0) return AS_OK;
    PhaseClock clk;
    const int64_t LG_CAP = (int64_t)1 << 26;
    int64_t max_N = 0;
    for (int64_t i = 0; i < n; ++i) {
        const int32_t* t = tables + i * 4;
        if (t[0] < 0 || t[1] < 0 || t[2] < 0 || t[3] < 0) return fail(AS_EINVAL, "table %lld has a negative count", (long long)i);
        const int64_t N = (int64_t)t[0] + t[1] + t[2] + t[3];
        if (N <= LG_CAP) max_N = std::max(max_N, N);
    }
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->exec_stream;
    if (max_N + 2 > c->lg_n) {  // extend the table: the host's own lgamma, a few threads
        const int64_t want = max_N + 2;
        std::vector<double> lg((size_t)want);
        const int nth = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(std::thread::hardware_concurrency(), 16u), want / 4096));
        auto work = [&](int k) {
            for (int64_t i = want * k / nth, e = want * (k + 1) / nth; i < e; ++i) {
                int sign = 0;
                lg[(size_t)i] = lgamma_r((double)i + 1.0, &sign);
            }
        };
        std::vector<std::thread> th;
        for (int k = 1; k < nth; ++k) th.emplace_back(work, k);
        work(0);
        for (auto& x : th) x.join();
        CU(c->lgtab.need((size_t)want * 8));
        CU(cudaMemcpy(c->lgtab.p, lg.data(), (size_t)want * 8, cudaMemcpyHostToDevice));
        c->lg_n = want;
    }
    clk.lap("fisher.lgamma_table");
    CU(c->misc.need((size_t)n * 24 + 64));
    int32_t* d_t = (int32_t*)c->misc.p;
    double* d_p = (double*)((char*)c->misc.p + (((size_t)n * 16 + 63) & ~(size_t)63));
    CU(cudaMemcpyAsync(d_t, tables, (size_t)n * 16, cudaMemcpyHostToDevice, st));
    std::vector<int64_t> on_host;  // tables beyond the lgamma table
    for (int64_t i = 0; i < n; ++i) {
        const int32_t* t = tables + i * 4;
        const int64_t N = (int64_t)t[0] + t[1] + t[2] + t[3];
        if (N > LG_CAP || N <= 170) on_host.push_back(i);  // beyond the table / Boost's factorial-table branch (as_fisher_test)
    }
    if (!on_host.empty()) {  // the kernel must not index past the table: give those warps an empty table
        std::vector<int32_t> zero(4, 0);
        for (int64_t i : on_host) CU(cudaMemcpyAsync(d_t + i * 4, zero.data(), 16, cudaMemcpyHostToDevice, st));
    }
    CU(as_launch_fisher(d_t, n, (const double*)c->lgtab.p, d_p, st));
    c->launches += 1;
    CU(cudaMemcpyAsync(p, d_p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int64_t i : on_host) p[i] = as_fisher_test(tables[i * 4], tables[i * 4 + 1], tables[i * 4 + 2], tables[i * 4 + 3]);
    clk.lap("fisher.device");
    return AS_OK;
}

int as_kf_gammaq_host(as_ctx* c, const double* s, const double* z, int64_t n, double* out) {
    if (!c || !s || !z || !out || n < 0) return fail(AS_EINVAL, "bad argument");
    if (n == 0) return AS_OK;
    CU(cudaSetDevice(c->device));
    CU(c->misc.need((size_t)n * 24));
    double* d_s = (double*)c->misc.p;
    double* d_z = d_s + n;
    double* d_o = d_z + n;
    cudaStream_t st = c->exec_stream;
    CU(cudaMemcpyAsync(d_s, s, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_z, z, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    CU(as_launch_gammaq(d_s, d_z, n, d_o, st));
    c->launches += 1;
    CU(cudaMemcpyAsync(out, d_o, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return AS_OK;
}

int as_synth_counts_dev(as_ctx* c, uint32_t* d_counts, int32_t n_samples, int64_t P, uint8_t* d_ref,
                        const as_synth_params* prm, void* stream) {
    if (!c || !d_counts || !prm || n_samples < 0 || P < 0) return fail(AS_EINVAL, "bad argument");
    CU(cudaSetDevice(c->device));
    CU(as_launch_synth(d_counts, n_samples, P, d_ref, prm, (cudaStream_t)stream));
    c->launches += 1;
    return AS_OK;
}

int as_synth_twin_links_dev(as_ctx* c, int64_t P, const as_synth_params* prm, int32_t* d_twin_next, int32_t* d_twin_head,
                            void* stream) {
    if (!c || !prm || !d_twin_next || !d_twin_head || P < 0) return fail(AS_EINVAL, "bad argument");
    if (prm->slot_offset % 125 != 0) return fail(AS_EINVAL, "slot_offset must be a multiple of the 125-slot amplicon");
    CU(cudaSetDevice(c->device));
    CU(as_launch_synth_twin_links(P, prm, d_twin_next, d_twin_head, (cudaStream_t)stream));
    c->launches += 1;
    return AS_OK;
}

}  // extern "C"
