// Deferred caller: the noise-floor sweep of BASELINE configs[3] (one pass over the tumour tensor for up to 8 threshold
// tables) as three kernels instead of one.
//
//   VC = source_codes/AmpliSolveVariantCalling.cpp.  Replaces, like call_staged_kernel, the row loop of callVariants
//   (VC:723-3296): strand counts, threshold lookup, mutationRulesPoissonQualityScore (VC:3834-3884) and the decision VC:898.
//
// Why three kernels.  ncu of the round-1 in-stage sweep kernel (profiles/r02_ncu_sweep_caller_before.txt): 8.05 ms for one
// 32 GB read = 50 % of the DRAM peak; the consumer warps sat on the scattered reads of the candidates' thresholds (five
// tables = 320 MB, beyond L2) and on the fp64 series WHILE HOLDING their shared-memory stage, so the producer had nothing
// to refill and the memory pipe ran dry after every candidate.  Here the streaming kernel does integer work only:
//
//   call_scan_kernel     TMA-staged scan (same ring as call_staged_kernel): coverage gate, alt != ref, integer pre-screen
//                        against the smallest threshold of all tables; the candidates -- a few per thousand (record, alt)
//                        pairs -- are compacted per warp into 24-byte entries and appended to a global list in batches
//                        (one atomic per ~25 entries).  No threshold read, no fp64, nothing long while a stage is held.
//   call_resolve_kernel  one thread per candidate: the thresholds of the candidate's (slot, alt) in every table (the list
//                        is in tile order, so these reads hit L2), the two exact screens per table (as_call.cuh) -> a bit
//                        mask of the tables in which the pair can still be a call; the survivors of table ci go to list ci
//                        (one atomic per table and 256-thread block).
//   call_series_kernel   grid.y = table: two lanes per survivor of that table's list (forward / reverse strand) evaluate the
//                        capped fp64 series of VC:3785-3794 -- every lane has work; calls are appended to the table's call
//                        list with one atomic per warp.
//
// Both lists live in scratch owned by the context.  An entry that does not fit its list is resolved on the spot by the
// thread that holds it (resolve_inline): slower, never wrong -- the call sets do not depend on the list capacities (tested
// with capacities of a few entries).
#include "as_kernels.h"

#include <cstdlib>

#include "as_call.cuh"
#include "as_pipeline.cuh"

namespace asdev {

struct Survivor {  // 32 bytes: an entry of one table's survivor list
    StagedCand c;
    uint32_t pad[2];
};
static_assert(sizeof(Survivor) == 32, "Survivor is two 16-byte words");

struct DeferredLists {
    StagedCand* cand;
    unsigned long long cap_cand;
    Survivor* surv;                // list of table ci at surv + ci * cap_surv
    unsigned long long cap_surv;   // per table
    unsigned long long* counters;  // [0] candidates appended (may exceed cap_cand), [1 + ci] survivors of table ci appended
};

struct CallSink {  // where calls go: table ci owns calls + ci * cap and n_calls[ci]
    const uint8_t* ref;
    const float* thr_view;
    int n_c;
    int64_t c_stride;
    as_call* calls;
    int64_t cap;
    unsigned long long* n_calls;
};

__device__ __forceinline__ void write_call(const CallSink& s, int ci, unsigned long long idx, const StagedCand& c, double p_fw,
                                           double p_bw) {
    if ((int64_t)idx >= s.cap) return;
    as_call o;
    o.sample = (int32_t)(c.sample_alt & 0x7ffffffu);
    o.slot = c.slot;
    o.alt = (int32_t)(c.sample_alt >> 30);
    o.ref = s.ref[c.slot];
    o.p_fw = p_fw; o.p_bw = p_bw;
    o.q_fw = q_from_p(p_fw); o.q_bw = q_from_p(p_bw);
    s.calls[(int64_t)ci * s.cap + (int64_t)idx] = o;
}

__device__ __forceinline__ float2 cand_thresholds(const CallSink& s, int ci, const StagedCand& c) {
    return *reinterpret_cast<const float2*>(s.thr_view + (int64_t)ci * s.c_stride + (int64_t)c.slot * 8 + 2 * (c.sample_alt >> 30));
}

// tables in which the pair survives both exact screens on both strands
__device__ __forceinline__ uint32_t screen_tables(const CallSink& s, const StagedCand& c) {
    uint32_t m = 0;
#pragma unroll
    for (int ci = 0; ci < 8; ++ci) {
        if (ci < s.n_c) {
            const float2 e = cand_thresholds(s, ci, c);
            m |= (strand_can_pass(c.k_fw, c.d_fw, e.x) && strand_can_pass(c.k_bw, c.d_bw, e.y)) ? (1u << ci) : 0u;
        }
    }
    return m;
}

// one thread, one candidate, every table in `tables`: the overflow path of both lists
__device__ __noinline__ void resolve_inline(const CallSink& s, const StagedCand& c, uint32_t tables) {
    for (int ci = 0; ci < s.n_c; ++ci) {
        if (!((tables >> ci) & 1u)) continue;
        const float2 e = cand_thresholds(s, ci, c);
        if (!(strand_can_pass(c.k_fw, c.d_fw, e.x) && strand_can_pass(c.k_bw, c.d_bw, e.y))) continue;
        const double pf = poisson_p((int)c.k_fw, (int)c.d_fw, e.x);  // VC:895
        if (!q_at_least_5(pf)) continue;
        const double pb = poisson_p((int)c.k_bw, (int)c.d_bw, e.y);  // VC:896
        if (!q_at_least_5(pb)) continue;                             // VC:898
        write_call(s, ci, atomicAdd(s.n_calls + ci, 1ull), c, pf, pb);
    }
}

#define AS_OUTQ_CAP 48 /* entries per warp; flushed before a round of 32 pushes could overflow it */

// append the n entries of a warp's queue (24-byte entries as uint2 words) to the candidate list
__device__ __forceinline__ void flush_candidates(const uint2* __restrict__ q, int n, const DeferredLists& L, const CallSink& s) {
    const int lane = threadIdx.x & 31;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(&L.counters[0], (unsigned long long)n);
    base = __shfl_sync(0xffffffffu, base, 0);
    const int n_fit = base >= L.cap_cand ? 0 : (int)min((unsigned long long)n, L.cap_cand - base);
    uint2* dst = reinterpret_cast<uint2*>(L.cand + base);
    for (int w = lane; w < n_fit * 3; w += 32) dst[w] = q[w];
    for (int i = n_fit + lane; i < n; i += 32) {  // list full: resolve here
        StagedCand c;
        const uint2 a = q[i * 3], b = q[i * 3 + 1], d = q[i * 3 + 2];
        c.k_fw = a.x; c.d_fw = a.y; c.k_bw = b.x; c.d_bw = b.y; c.sample_alt = d.x; c.slot = (int32_t)d.y;
        resolve_inline(s, c, 0xffu);
    }
    __syncwarp();
}

template <int K, int STAGES>
__global__ void __launch_bounds__(AS_CTA_THREADS, 7)
call_scan_kernel(const uint4* __restrict__ counts, int T, int64_t P, int64_t p0, int64_t p1, int chunk, uint32_t cut,
                 DeferredLists L, CallSink sink) {
    static_assert(K * 4 <= 32, "candidate mask is one 32-bit word per thread and stage");
    constexpr int CAND_CAP = K * 32 * 3;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * STAGES];
    __shared__ uint16_t cand_all[AS_CONSUMER_WARPS][CAND_CAP];
    __shared__ __align__(8) uint2 outq_all[AS_CONSUMER_WARPS][AS_OUTQ_CAP * 3];
    StageRing<K, STAGES> ring;
    ring.init(smem_raw, bars);
    const int64_t tile0 = p0 + (int64_t)blockIdx.x * AS_TILE_SLOTS;
    const int n_slots = (int)min((int64_t)AS_TILE_SLOTS, p1 - tile0);
    const int t0 = blockIdx.y * chunk, t1 = min(T, t0 + chunk);
    const int tid = threadIdx.x;
    if (tid >= AS_TILE_SLOTS) {  // producer warp
        if (tid == AS_TILE_SLOTS) ring.produce(counts + tile0, 2 * P, P, t0, t1, n_slots);
        return;
    }
    const int lane = tid & 31, warp = tid >> 5;
    const int64_t p = tile0 + tid;
    uint32_t notref = 0;
    uint32_t Rf = 0, Rb = 0;  // floor(e_min * 2^32) per strand over the callable alt bases and all tables; 0 screens nothing
    if (tid < n_slots) {
        const uint32_t r = sink.ref[p];
        if (r <= 3) {
            notref = 0xfu & ~(1u << r);
            Rf = Rb = 0xFFFFFFFFu;
            for (int ci = 0; ci < sink.n_c; ++ci) {
                const float4 a = *reinterpret_cast<const float4*>(sink.thr_view + ci * sink.c_stride + p * 8);
                const float4 b = *reinterpret_cast<const float4*>(sink.thr_view + ci * sink.c_stride + p * 8 + 4);
                const float e[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if ((uint32_t)i == r) continue;
#pragma unroll
                    for (int st = 0; st < 2; ++st) {
                        const float raw = e[2 * i + st];
                        if (raw == -1.0f) continue;  // no threshold: never a call (VC:3844-3849), no bound on the minimum
                        const float ee = effective_err(raw);
                        // e * 2^32 is exact and < 2^32 for 0 < e < 1; anything else switches the pre-screen off for the strand
                        const uint32_t R = (ee > 0.0f && ee < 1.0f) ? __float2uint_rz(ee * 4294967296.0f) : 0u;
                        if (st == 0) Rf = min(Rf, R); else Rb = min(Rb, R);
                    }
                }
            }
        }
    }
    uint16_t* cand = cand_all[warp];
    uint2* outq = outq_all[warp];
    int n_q = 0;  // warp-uniform
    uint32_t notref_rep = notref;
#pragma unroll
    for (int j = 1; j < K; ++j) notref_rep |= notref << (4 * j);

    int it = 0;
    for (int t = t0; t < t1; t += K, ++it) {
        const uint4* st = ring.consumer_wait(it);
        const int k = min(K, t1 - t);
        // ---- scan: integer tests only (coverage gate VC:898, alt != ref, pre-screen; k == 0 -> Q = 0 VC:3858-3861)
        uint32_t mask = 0;
#pragma unroll
        for (int j = 0; j < K; ++j) {
            if (j < k) {
                const uint4 fw = st[(j * 2 + 0) * AS_TILE_SLOTS + tid];
                const uint4 bw = st[(j * 2 + 1) * AS_TILE_SLOTS + tid];
                const uint32_t FW = fw.x + fw.y + fw.z + fw.w, BW = bw.x + bw.y + bw.z + bw.w;
                const uint32_t mf = prescreen_k(FW, Rf), mb = prescreen_k(BW, Rb);
                const uint32_t m = ((fw.x > mf && bw.x > mb) ? 1u : 0u) | ((fw.y > mf && bw.y > mb) ? 2u : 0u) |
                                   ((fw.z > mf && bw.z > mb) ? 4u : 0u) | ((fw.w > mf && bw.w > mb) ? 8u : 0u);
                const bool ok = (int32_t)fw.x >= 0 && min(FW, BW) >= cut;
                mask |= (ok ? m : 0u) << (4 * j);
            }
        }
        mask &= notref_rep;
        if (__ballot_sync(0xffffffffu, mask != 0) != 0) {
            // ---- compact the candidates of this stage: one prefix sum per warp and stage
            const int mine = __popc(mask);
            int incl = mine;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int up = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += up;
            }
            const int total = __shfl_sync(0xffffffffu, incl, 31);
            int off = incl - mine;
            uint32_t mm = mask;
            while (mm) {
                const int bit = __ffs(mm) - 1;
                mm &= mm - 1;
                cand[off++] = (uint16_t)((bit << 5) | lane);
            }
            __syncwarp();
            // ---- full warps turn the references into entries (counts re-read from the resident stage) and queue them
            for (int base = 0; base < total; base += 32) {
                if (n_q + 32 > AS_OUTQ_CAP) { flush_candidates(outq, n_q, L, sink); n_q = 0; }
                const int i = base + lane;
                if (i < total) {
                    const uint32_t e = cand[i];
                    const int src = e & 31, bit = e >> 5, j = bit >> 2, b = bit & 3;
                    const int col = warp * 32 + src;
                    const uint4 fw = st[(j * 2 + 0) * AS_TILE_SLOTS + col];
                    const uint4 bw = st[(j * 2 + 1) * AS_TILE_SLOTS + col];
                    uint2* dst = outq + (n_q + lane) * 3;
                    dst[0] = make_uint2(comp(fw, b), fw.x + fw.y + fw.z + fw.w);
                    dst[1] = make_uint2(comp(bw, b), bw.x + bw.y + bw.z + bw.w);
                    dst[2] = make_uint2((uint32_t)(t + j) | ((uint32_t)b << 30), (uint32_t)(tile0 + col));
                }
                n_q += min(32, total - base);
                __syncwarp();
            }
        }
        ring.consumer_release(it);
    }
    if (n_q > 0) flush_candidates(outq, n_q, L, sink);
}

__global__ void __launch_bounds__(256)
call_resolve_kernel(DeferredLists L, CallSink sink) {
    __shared__ uint32_t warp_n[8][8];  // [table][warp]
    __shared__ unsigned long long block_base[8];
    const unsigned long long n = min(L.counters[0], L.cap_cand);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t below = (1u << lane) - 1u;
    for (unsigned long long i0 = (unsigned long long)blockIdx.x * 256; i0 < n; i0 += (unsigned long long)gridDim.x * 256) {
        const unsigned long long i = i0 + threadIdx.x;
        StagedCand c;
        uint32_t tables = 0;
        if (i < n) {
            const uint2* src = reinterpret_cast<const uint2*>(L.cand + i);
            const uint2 a = src[0], b = src[1], d = src[2];
            c.k_fw = a.x; c.d_fw = a.y; c.k_bw = b.x; c.d_bw = b.y; c.sample_alt = d.x; c.slot = (int32_t)d.y;
            tables = screen_tables(sink, c);
        }
        uint32_t rank = 0;  // rank of this lane among its warp's survivors of table ci: 5 bits per table, tables 0..5 here, 6..7 in rank_hi
        uint32_t rank_hi = 0;
#pragma unroll
        for (int ci = 0; ci < 8; ++ci) {
            if (ci < sink.n_c) {
                const unsigned votes = __ballot_sync(0xffffffffu, (tables >> ci) & 1u);
                if (lane == 0) warp_n[ci][warp] = __popc(votes);
                const uint32_t r = __popc(votes & below);
                if (ci < 6) rank |= r << (5 * ci); else rank_hi |= r << (5 * (ci - 6));
            }
        }
        __syncthreads();
        if (threadIdx.x < sink.n_c) {
            uint32_t tot = 0;
            for (int w = 0; w < 8; ++w) tot += warp_n[threadIdx.x][w];
            block_base[threadIdx.x] = tot ? atomicAdd(&L.counters[1 + threadIdx.x], (unsigned long long)tot) : 0ull;
        }
        __syncthreads();
        if (tables != 0) {
            uint32_t inline_tables = 0;
#pragma unroll
            for (int ci = 0; ci < 8; ++ci) {
                if (ci < sink.n_c && ((tables >> ci) & 1u)) {
                    unsigned long long idx = block_base[ci] + ((ci < 6 ? rank >> (5 * ci) : rank_hi >> (5 * (ci - 6))) & 31u);
                    for (int w = 0; w < warp; ++w) idx += warp_n[ci][w];
                    if (idx < L.cap_surv) {
                        uint4* dst = reinterpret_cast<uint4*>(L.surv + (unsigned long long)ci * L.cap_surv + idx);
                        dst[0] = make_uint4(c.k_fw, c.d_fw, c.k_bw, c.d_bw);
                        dst[1] = make_uint4(c.sample_alt, (uint32_t)c.slot, 0u, 0u);
                    } else {
                        inline_tables |= 1u << ci;  // list full: resolve here
                    }
                }
            }
            if (inline_tables) resolve_inline(sink, c, inline_tables);
        }
        __syncthreads();  // warp_n / block_base are rewritten by the next round
    }
}

__global__ void __launch_bounds__(128)
call_series_kernel(DeferredLists L, CallSink sink) {
    const int ci = blockIdx.y;
    const unsigned long long n = min(L.counters[1 + ci], L.cap_surv);
    const Survivor* list = L.surv + (unsigned long long)ci * L.cap_surv;
    const int lane = threadIdx.x & 31, pair = lane >> 1, strand = lane & 1;
    const unsigned long long warps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    for (unsigned long long g = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; g * 16 < n; g += warps) {
        const unsigned long long i = g * 16 + pair;
        StagedCand c;
        const bool active = i < n;
        double p = 1.0;
        if (active) {
            const uint4* src = reinterpret_cast<const uint4*>(list + i);
            const uint4 a = src[0], b = src[1];
            c.k_fw = a.x; c.d_fw = a.y; c.k_bw = a.z; c.d_bw = a.w; c.sample_alt = b.x; c.slot = (int32_t)b.y;
            const float e = sink.thr_view[(int64_t)ci * sink.c_stride + (int64_t)c.slot * 8 + 2 * (c.sample_alt >> 30) + strand];
            p = strand == 0 ? poisson_p((int)c.k_fw, (int)c.d_fw, e) : poisson_p((int)c.k_bw, (int)c.d_bw, e);  // VC:895-896
        }
        const double p_other = __shfl_xor_sync(0xffffffffu, p, 1);
        const bool is_call = active && strand == 0 && q_at_least_5(p) && q_at_least_5(p_other);  // VC:898
        const unsigned votes = __ballot_sync(0xffffffffu, is_call);
        if (votes == 0) continue;
        const int leader = __ffs(votes) - 1;
        unsigned long long base = 0;
        if (lane == leader) base = atomicAdd(sink.n_calls + ci, (unsigned long long)__popc(votes));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (is_call) write_call(sink, ci, base + __popc(votes & ((1u << lane) - 1u)), c, p, p_other);
    }
}

}  // namespace asdev

using namespace asdev;

size_t as_deferred_scratch_bytes(int T, int64_t n_slots, int64_t cap_override, int64_t* cap_cand, int64_t* cap_surv) {
    // candidates: a few per thousand (record, alt) pairs on real panels; room for one record in 24, within 1 Mi .. 64 Mi
    // entries (1.5 GB).  Survivors: a quarter of that.  Whatever does not fit is resolved inline by the kernels.
    // cap_override > 0 sets the candidate capacity (a quarter of it, at least 1, for the survivors): the scratch is sized
    // for the capacities in use, whichever way they were chosen.
    int64_t cc = (int64_t)T * n_slots / 24;
    cc = cap_override > 0 ? cap_override : std::max<int64_t>(1 << 20, std::min<int64_t>(cc, 64ll << 20));
    *cap_cand = cc;
    *cap_surv = cap_override > 0 ? std::max<int64_t>(1, cc / 4) : std::max<int64_t>(1 << 18, cc / 4);  // per table
    return 4096 + (size_t)cc * sizeof(StagedCand) + 8 * (size_t)*cap_surv * sizeof(Survivor) + 512 * AS_DEFER_MAX_CHUNKS;
}

// pieces a range is cut into: at most `want`, and at least two full waves of scan CTAs (148 SMs x 7) per piece
int as_deferred_chunks(int64_t n_slots, int want) {
    const int64_t tiles = (n_slots + AS_TILE_SLOTS - 1) / AS_TILE_SLOTS;
    return (int)std::max<int64_t>(1, std::min<int64_t>(std::min(want, AS_DEFER_MAX_CHUNKS), tiles / (148 * 7 * 2)));
}

// d_scratch: as_deferred_scratch_bytes() bytes, 256-byte aligned: counters | candidates | survivors.
// The slot range is cut into n_chunks pieces (each with its share of the two lists): the scan of piece i+1 runs on `st`
// while the resolve and series kernels of piece i run on `aux` (a high-priority stream; ev[i] orders them) -- the scan is
// bound by HBM, the series by the fp64 pipe, so the two overlap almost for free.  n_chunks == 1: everything on `st`.
// Launches: 1 memset + 3 kernels per piece.
cudaError_t as_launch_call_deferred(const uint32_t* d_counts, int T, int64_t P, int64_t p0, int64_t p1, const uint8_t* d_ref,
                                    const float* d_thr_views, int n_c, int64_t c_stride, uint32_t cut, as_call* d_calls,
                                    int64_t cap, unsigned long long* d_n_calls, void* d_scratch, int64_t cap_cand,
                                    int64_t cap_surv, cudaStream_t st, cudaStream_t aux, cudaEvent_t* ev, int n_chunks) {
    if (p1 <= p0 || T <= 0 || n_c <= 0) return cudaSuccess;
    if (n_c > 8) return cudaErrorInvalidValue;
    const int64_t tiles = (p1 - p0 + AS_TILE_SLOTS - 1) / AS_TILE_SLOTS;
    n_chunks = (aux == nullptr || ev == nullptr) ? 1 : as_deferred_chunks(p1 - p0, n_chunks);
    CallSink sink{d_ref, d_thr_views, n_c, c_stride, d_calls, cap, d_n_calls};
    unsigned long long* counters = (unsigned long long*)d_scratch;  // 16 per piece: candidates, survivors of tables 0..7
    StagedCand* cand0 = (StagedCand*)((char*)d_scratch + 4096);
    Survivor* surv0 = (Survivor*)((char*)d_scratch + 4096 + (((size_t)cap_cand * sizeof(StagedCand) + 255) & ~(size_t)255));
    cudaError_t e = cudaMemsetAsync(counters, 0, 128 * AS_DEFER_MAX_CHUNKS, st);
    if (e != cudaSuccess) return e;
    // ring geometry of the scan kernel (samples per stage, stages); five tables on the c3 shard: 0 = (3,2) 5.65 ms, 1 = (4,2)
    // 5.62, 2 = (3,3) 5.59 (default), 3 = (2,3) 5.62.  AS_SCAN_GEOM selects another one (experiments).
    static int geom = -1;
    if (geom < 0) { const char* g = getenv("AS_SCAN_GEOM"); geom = g ? (atoi(g) & 3) : 2; }
    int smem = 0;
    {
        static bool configured[AS_MAX_DEVICES][4] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        const void* fn = geom == 1 ? (const void*)call_scan_kernel<4, 2> : geom == 2 ? (const void*)call_scan_kernel<3, 3>
                         : geom == 3 ? (const void*)call_scan_kernel<2, 3> : (const void*)call_scan_kernel<3, 2>;
        smem = geom == 1 ? StageRing<4, 2>::kStageBytes * 2 : geom == 2 ? StageRing<3, 3>::kStageBytes * 3
               : geom == 3 ? StageRing<2, 3>::kStageBytes * 3 : StageRing<3, 2>::kStageBytes * 2;
        if (dev < 0 || dev >= AS_MAX_DEVICES || !configured[dev][geom & 3]) {
            e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            if (e != cudaSuccess) return e;
            if (dev >= 0 && dev < AS_MAX_DEVICES) configured[dev][geom & 3] = true;
        }
    }
    const int chunk = as_call_chunk(T, p1 - p0);
    const unsigned gy = (unsigned)((T + chunk - 1) / chunk);
    for (int ch = 0; ch < n_chunks; ++ch) {
        const int64_t t_lo = tiles * ch / n_chunks, t_hi = tiles * (ch + 1) / n_chunks;
        const int64_t q0 = p0 + t_lo * AS_TILE_SLOTS, q1 = std::min(p1, p0 + t_hi * AS_TILE_SLOTS);
        if (q1 <= q0) continue;
        DeferredLists L;
        L.counters = counters + 16 * ch;
        L.cap_cand = (unsigned long long)(cap_cand / n_chunks);
        L.cap_surv = (unsigned long long)(cap_surv / n_chunks);
        L.cand = cand0 + (size_t)ch * L.cap_cand;
        L.surv = surv0 + (size_t)ch * 8 * L.cap_surv;
        dim3 grid((unsigned)(t_hi - t_lo), gy);
#define AS_SCAN_LAUNCH(KK, SS) call_scan_kernel<KK, SS><<<grid, AS_CTA_THREADS, smem, st>>>(reinterpret_cast<const uint4*>(d_counts), T, P, q0, q1, chunk, cut, L, sink)
        if (geom == 1) AS_SCAN_LAUNCH(4, 2); else if (geom == 2) AS_SCAN_LAUNCH(3, 3); else if (geom == 3) AS_SCAN_LAUNCH(2, 3); else AS_SCAN_LAUNCH(3, 2);
#undef AS_SCAN_LAUNCH
        cudaStream_t post = st;
        if (n_chunks > 1) {
            if ((e = cudaEventRecord(ev[ch], st)) != cudaSuccess) return e;
            if ((e = cudaStreamWaitEvent(aux, ev[ch], 0)) != cudaSuccess) return e;
            post = aux;
        }
        call_resolve_kernel<<<148 * 8, 256, 0, post>>>(L, sink);
        call_series_kernel<<<dim3(148 * 4, (unsigned)n_c), 128, 0, post>>>(L, sink);
    }
    if (n_chunks > 1) {  // join: control returns to `st` when the last series kernel is done
        if ((e = cudaEventRecord(ev[n_chunks], aux)) != cudaSuccess) return e;
        if ((e = cudaStreamWaitEvent(st, ev[n_chunks], 0)) != cudaSuccess) return e;
    }
    return cudaGetLastError();
}
