// CUDA kernels of the AmpliSolve hot path for sm_100a, and their launchers.
//
//   EE = source_codes/AmpliSolveErrorEstimation.cpp, VC = source_codes/AmpliSolveVariantCalling.cpp
//
// Both kernels are scans over a dense count tensor uint32 [sample][strand][slot][base]: one 16-byte
// word per (sample, strand, slot), so a warp covering 32 consecutive slots reads 512 contiguous bytes
// per (sample, strand) with one LDG.128 per lane.  Nothing here is a dense contraction: no tensor
// cores.  The bound is HBM (32 algorithmic bytes per record); the instruction budget at the roofline
// is ~150 issue slots per record, which is why the filter arithmetic is division-free (as_noise.cuh)
// and why the caller screens records with integer tests and only evaluates the fp64 incomplete-gamma
// series for the rare survivors, compacted through per-warp shared-memory queues so that the fp64
// loops run on full warps.
#include "as_kernels.h"

#include "as_device.cuh"
#include "as_noise.cuh"
#include "as_pipeline.cuh"
#include "as_call.cuh"

namespace asdev {

// ------------------------------------------------------------------------------------------------
// noise model, singleton slots: one thread per slot, all normals in sequence
// ------------------------------------------------------------------------------------------------
template <int UNROLL>
__global__ void __launch_bounds__(AS_NOISE_THREADS)
noise_main_kernel(const uint4* __restrict__ counts, int S, int64_t P, int64_t p0, int64_t p1,
                  const int32_t* __restrict__ twin_next, const int32_t* __restrict__ twin_head, int64_t twin_base,
                  float C, uint32_t cut, float* __restrict__ thr, float* __restrict__ germ_val,
                  uint8_t* __restrict__ germ_state, uint32_t* __restrict__ count, uint32_t* __restrict__ nrec) {
    const int64_t p = p0 + (int64_t)blockIdx.x * AS_NOISE_THREADS + threadIdx.x;
    if (p >= p1) return;
    // members of a twin group (position enumerated by overlapping amplicons) are done by noise_twin_kernel;
    // twin_head holds panel-global slot ids, p + twin_base is this slot's
    if (twin_next != nullptr && (twin_next[p] >= 0 || twin_head[p] != (int32_t)(p + twin_base))) return;

    const uint4* q = counts + p;
    const int64_t sstride = 2 * P;  // uint4 words per sample
    NoiseAcc acc;
    FastAcc f;
    fast_init(f);
    for (int sb = 0; sb < S; sb += AS_FOLD_EVERY) {
        const int se = min(S, sb + AS_FOLD_EVERY);
        int s = sb;
        for (; s + UNROLL <= se; s += UNROLL) {
            uint4 fw[UNROLL], bw[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                fw[u] = ld_stream(q + (int64_t)(s + u) * sstride);
                bw[u] = ld_stream(q + (int64_t)(s + u) * sstride + P);
            }
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) fast_accumulate(f, fw[u], bw[u], C, cut);
        }
        for (; s < se; ++s) {
            const uint4 fw = ld_stream(q + (int64_t)s * sstride);
            const uint4 bw = ld_stream(q + (int64_t)s * sstride + P);
            fast_accumulate(f, fw, bw, C, cut);
        }
        fast_fold(f);
    }
    if (f.big < (1u << 24)) {
        fast_to_general(f, acc);
    } else {
        // some record of this slot has a depth of 2^24 or more: int -> float is inexact there, redo the slot
        // with the general code (never seen in practice; keeps the result exact for every uint32 input)
        noise_init(acc);
#pragma unroll 1
        for (int s = 0; s < S; ++s) {
            const uint4 fw = ld_stream(q + (int64_t)s * sstride);
            const uint4 bw = ld_stream(q + (int64_t)s * sstride + P);
            noise_accumulate<false>(acc, fw, bw, C, cut);
        }
    }
    noise_store(acc, p, thr, germ_val, germ_state, count, nrec);
}

// A duplicated position whose two slots lie in the same 128-slot CTA tile (the common case: consecutive amplicons
// overlapping by a few bases put the second enumeration `overlap` slots after the first) is reduced by the thread of
// its first slot, which reads both records of every sample in file order.  Returns the distance to the twin slot
// for such a head, 0 otherwise.  idx = index into the twin arrays, gid = panel-global id of that slot, tid = index in
// the CTA tile, n_slots = valid slots of the tile.  Everything else with twins goes to noise_twin_kernel.
__device__ __forceinline__ int intile_twin_distance(const int32_t* __restrict__ twin_next,
                                                    const int32_t* __restrict__ twin_head, int64_t idx, int64_t gid, int tid,
                                                    int n_slots) {
    const int32_t nx = twin_next[idx];
    if (nx < 0 || twin_head[idx] != (int32_t)gid) return 0;
    const int64_t d = (int64_t)nx - gid;
    if (d <= 0 || tid + d >= n_slots) return 0;
    if (twin_next[idx + d] >= 0) return 0;  // three or more enumerations: general kernel
    return (int)d;
}

// Finalise one slot: fast-path state, or the general code over global memory when a depth >= 2^24 was seen.
// twin_d > 0: the slot at distance twin_d belongs to the same position (its rows follow this slot's, per sample).
__device__ __forceinline__ void noise_finish_slot(FastAcc& f, const uint4* __restrict__ q, int S, int64_t P, float C,
                                                  uint32_t cut, int64_t p, int twin_d, float* __restrict__ thr,
                                                  float* __restrict__ germ_val, uint8_t* __restrict__ germ_state,
                                                  uint32_t* __restrict__ count, uint32_t* __restrict__ nrec) {
    NoiseAcc acc;
    if (f.big < (1u << 24)) {
        fast_to_general(f, acc);
    } else {
        noise_init(acc);
#pragma unroll 1
        for (int s = 0; s < S; ++s) {
#pragma unroll 1
            for (int r = 0; r <= (twin_d > 0 ? 1 : 0); ++r) {
                const uint4 fw = ld_stream(q + (int64_t)s * 2 * P + r * twin_d);
                const uint4 bw = ld_stream(q + (int64_t)s * 2 * P + P + r * twin_d);
                noise_accumulate<false>(acc, fw, bw, C, cut);
            }
        }
    }
    noise_store(acc, p, thr, germ_val, germ_state, count, nrec);
    if (twin_d > 0) noise_store(acc, p + twin_d, thr, germ_val, germ_state, count, nrec);
}

// ------------------------------------------------------------------------------------------------
// noise model, singleton slots, TMA-staged: producer warp + 4 consumer warps (as_pipeline.cuh)
// ------------------------------------------------------------------------------------------------
template <int K, int STAGES>
__global__ void __launch_bounds__(AS_CTA_THREADS, 4)
noise_staged_kernel(const uint4* __restrict__ counts, int S, int64_t P, int64_t p0, int64_t p1,
                    const int32_t* __restrict__ twin_next, const int32_t* __restrict__ twin_head, int64_t twin_base,
                    float C, uint32_t cut, float* __restrict__ thr, float* __restrict__ germ_val,
                    uint8_t* __restrict__ germ_state, uint32_t* __restrict__ count, uint32_t* __restrict__ nrec) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * STAGES];
    StageRing<K, STAGES> ring;
    ring.init(smem_raw, bars);
    const int64_t tile0 = p0 + (int64_t)blockIdx.x * AS_TILE_SLOTS;
    const int n_slots = (int)min((int64_t)AS_TILE_SLOTS, p1 - tile0);
    const int tid = threadIdx.x;
    if (tid >= AS_TILE_SLOTS) {  // producer warp
        if (tid == AS_TILE_SLOTS) ring.produce(counts + tile0, 2 * P, P, 0, S, n_slots);
        return;
    }
    const int64_t p = tile0 + tid;
    bool active = tid < n_slots;
    // role of this slot: 0 singleton, 1 first slot of a twin pair whose second slot is in this CTA tile, 2 that second
    // slot, 3 any other member of a twin group (left to noise_pair_kernel / noise_twin_kernel)
    int role = 0, twin_d = 0;
    constexpr bool kPairsInTile = AS_INTILE_TWINS && (StageRing<K, STAGES>::kStageBytes * STAGES >= AS_TILE_SLOTS * (int)sizeof(PairXfer));
    if (active && twin_next != nullptr) {
        const int64_t gid = p + twin_base;
        if (twin_next[p] >= 0 || twin_head[p] != (int32_t)gid) role = 3;
        if (kPairsInTile) {
            twin_d = intile_twin_distance(twin_next, twin_head, p, gid, tid, n_slots);
            if (twin_d > 0) {
                role = 1;
            } else if (role == 3) {
                const int64_t back = gid - (int64_t)twin_head[p];  // distance to the head of this slot's group
                if (back > 0 && back <= tid && intile_twin_distance(twin_next, twin_head, p - back, gid - back, tid - (int)back, n_slots) == (int)back)
                    role = 2;
            }
        }
        if (role == 3) active = false;
    }

    FastAcc f;
    fast_init(f);
    int it = 0, since_fold = 0;
    for (int t = 0; t < S; t += K, ++it) {
        const uint4* st = ring.consumer_wait(it);
        const int k = min(K, S - t);
        if (active) {
#pragma unroll
            for (int j = 0; j < K; ++j) {
                if (j < k) {
                    const uint4 fw = st[(j * 2 + 0) * AS_TILE_SLOTS + tid];
                    const uint4 bw = st[(j * 2 + 1) * AS_TILE_SLOTS + tid];
                    fast_accumulate(f, fw, bw, C, cut);
                }
            }
        }
        ring.consumer_release(it);
        since_fold += K;
        if (since_fold >= AS_FOLD_EVERY) { fast_fold(f); since_fold = 0; }
    }
    fast_fold(f);

    if (kPairsInTile && twin_next != nullptr) {
        // Twin pairs inside the tile: both threads reduced their own rows like singletons (no cost in the loop above);
        // the second slot's thread hands its state over through the (now idle) ring memory and the first slot's thread
        // merges EXACTLY: sums add; for Germ_Max the file order is (sample, first slot) < (sample, second slot), the
        // overall first qualifying record is dropped and the other thread's first one joins the maximum (pair_merge).
        PairXfer* xfer = reinterpret_cast<PairXfer*>(smem_raw);
        PairFirst mine;
        if (role == 1 || role == 2) pair_find_first(mine, f, counts + p, S, P, C, cut);
        asm volatile("bar.sync 1, %0;" ::"n"(AS_TILE_SLOTS) : "memory");  // every consumer warp is done with the ring
        if (role == 2) { xfer[tid].f = f; xfer[tid].first = mine; }
        asm volatile("bar.sync 1, %0;" ::"n"(AS_TILE_SLOTS) : "memory");
        if (role == 1) pair_merge(f, mine, xfer[tid + twin_d].f, xfer[tid + twin_d].first);
        if (role == 2) active = false;  // stored by the first slot's thread
    }
    if (active) noise_finish_slot(f, counts + p, S, P, C, cut, p, role == 1 ? twin_d : 0, thr, germ_val, germ_state, count, nrec);
}

// ------------------------------------------------------------------------------------------------
// noise model, twin groups: the reference keys records by "chrom_pos" text, so every row of every
// slot of a duplicated position feeds ONE estimate (EE:1241-1245), in the order file, then row.
// ------------------------------------------------------------------------------------------------
// Heads of twin groups in [p0, p1): 2-chains (a position enumerated twice, by far the common case) go to the pair
// list, longer chains to the general list.  counters[0] = pairs, counters[1] = longer groups.
__global__ void twin_heads_kernel(const int32_t* __restrict__ twin_next, const int32_t* __restrict__ twin_head,
                                  int64_t p0, int64_t p1, int skip_intile, int32_t* __restrict__ pairs,
                                  int32_t* __restrict__ groups, uint32_t* __restrict__ counters) {
    const int64_t p = p0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= p1) return;
    const int32_t nx = twin_next[p];
    if (twin_head[p] != (int32_t)p || nx < 0) return;
    if (skip_intile) {  // pairs inside one CTA tile of the staged kernel are reduced there
        const int tid = (int)((p - p0) % AS_TILE_SLOTS);
        const int n_slots = (int)min((int64_t)AS_TILE_SLOTS, p1 - (p - tid));
        if (intile_twin_distance(twin_next, twin_head, p, p, tid, n_slots) > 0) return;
    }
    if (twin_next[nx] < 0)
        pairs[atomicAdd(&counters[0], 1u)] = (int32_t)p;
    else
        groups[atomicAdd(&counters[1], 1u)] = (int32_t)p;
}

// Twin pairs: a warp takes eight pairs, four lanes per pair (one per base), and walks the samples in file order (slot
// a's row, then slot b's row) with the fast-path arithmetic -- no partial-state merge.  The 32 lanes first fetch the
// 4 words (fw/bw of a and b) x 8 pairs of AS_PAIR_BATCH samples into a per-warp shared-memory block, so that
// AS_PAIR_BATCH scattered 16-byte reads per lane are in flight at once; then every lane reads its pair's four words
// back (broadcast within the quad).
#define AS_PAIR_BATCH 8
__global__ void __launch_bounds__(128)
noise_pair_kernel(const uint4* __restrict__ counts, int S, int64_t P, const int32_t* __restrict__ twin_next,
                  const int32_t* __restrict__ pairs, const uint32_t* __restrict__ counters, float C, uint32_t cut,
                  float* __restrict__ thr, float* __restrict__ germ_val, uint8_t* __restrict__ germ_state,
                  uint32_t* __restrict__ count, uint32_t* __restrict__ nrec) {
    __shared__ __align__(16) uint4 stage_all[4][AS_PAIR_BATCH][32];
    const int lane = threadIdx.x & 31, base = lane & 3, quad0 = lane & ~3;
    uint4 (*stage)[32] = stage_all[threadIdx.x >> 5];
    const uint32_t n = counters[0];
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const int64_t sstride = 2 * P;
    for (uint32_t wg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; wg * 8 < n; wg += warps) {
        const uint32_t g = wg * 8 + (lane >> 2);
        const bool valid = g < n;
        const int32_t a = valid ? pairs[g] : 0;
        const int32_t b = valid ? twin_next[a] : 0;
        // this lane fetches word `base` of its pair: 0 = fw(a), 1 = bw(a), 2 = fw(b), 3 = bw(b)
        const uint4* src = counts + ((base & 2) ? b : a) + ((base & 1) ? P : 0);
        FastBase f;
        f.s_b_fw = f.s_b_bw = 0u;
        f.s_d_fw = f.s_d_bw = f.s_p_fw = f.s_p_bw = 0.0;
        f.count = 0u; f.g_x = 1u; f.g_rd = 0u;
        uint32_t n_records = 0, big = 0;
        int since_fold = 0;
        for (int s0 = 0; s0 < S; s0 += AS_PAIR_BATCH) {
            const int k = min(AS_PAIR_BATCH, S - s0);
            uint4 w[AS_PAIR_BATCH];
#pragma unroll
            for (int j = 0; j < AS_PAIR_BATCH; ++j)
                if (j < k && valid) w[j] = ld_stream(src + (int64_t)(s0 + j) * sstride);
            __syncwarp();  // the previous batch has been consumed
#pragma unroll
            for (int j = 0; j < AS_PAIR_BATCH; ++j)
                if (j < k && valid) stage[j][lane] = w[j];
            __syncwarp();
            if (valid) {
#pragma unroll 2
                for (int j = 0; j < k; ++j) {
#pragma unroll
                    for (int row = 0; row < 2; ++row) {
                        const uint4 fw = stage[j][quad0 + 2 * row], bw = stage[j][quad0 + 2 * row + 1];
                        if ((int32_t)fw.x >= 0) {
                            FastRecord r;
                            n_records += 1;
                            fast_record(r, fw, bw, C, cut);
                            big |= r.RD;
                            fast_base_update(f, r, comp(fw, base), comp(bw, base));
                        }
                    }
                }
            }
            since_fold += 2 * AS_PAIR_BATCH;
            if (since_fold >= AS_FOLD_EVERY) {
                f.s_p_fw = __dadd_rn(f.s_p_fw, u32_to_double(f.s_b_fw));
                f.s_p_bw = __dadd_rn(f.s_p_bw, u32_to_double(f.s_b_bw));
                f.s_b_fw = f.s_b_bw = 0u;
                since_fold = 0;
            }
        }
        const bool redo = valid && big >= (1u << 24);
        if (redo && base == 0) {
            // a depth of 2^24 or more: int -> float is inexact, the lane of base A redoes the pair with the general code
            NoiseAcc acc;
            noise_init(acc);
            const uint4 *qa = counts + a, *qb = counts + b;
#pragma unroll 1
            for (int s = 0; s < S; ++s) {
                noise_accumulate<false>(acc, ld_stream(qa + (int64_t)s * sstride), ld_stream(qa + (int64_t)s * sstride + P), C, cut);
                noise_accumulate<false>(acc, ld_stream(qb + (int64_t)s * sstride), ld_stream(qb + (int64_t)s * sstride + P), C, cut);
            }
            noise_store(acc, a, thr, germ_val, germ_state, count, nrec);
            noise_store(acc, b, thr, germ_val, germ_state, count, nrec);
        }
        NoiseBase nb;
        fast_base_to_general(f, nb);
        float q_fw, q_bw, gv;
        uint32_t st;
        noise_final_base(nb, n_records, base, q_fw, q_bw, gv, st);
        // gather the four bases on the quad's first lane
        float t[8], gg[4];
        uint32_t c[4], gs = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            t[2 * i] = __shfl_sync(0xffffffffu, q_fw, quad0 + i);
            t[2 * i + 1] = __shfl_sync(0xffffffffu, q_bw, quad0 + i);
            gg[i] = __shfl_sync(0xffffffffu, gv, quad0 + i);
            c[i] = __shfl_sync(0xffffffffu, nb.count, quad0 + i);
            gs |= __shfl_sync(0xffffffffu, st, quad0 + i) << (8 * i);
        }
        if (valid && !redo && base == 0) {
            noise_store_raw(a, t, gg, gs, c, n_records, thr, germ_val, germ_state, count, nrec);
            noise_store_raw(b, t, gg, gs, c, n_records, thr, germ_val, germ_state, count, nrec);
        }
    }
}

__device__ __forceinline__ uint32_t shfl_down_u32(uint32_t v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
__device__ __forceinline__ unsigned long long shfl_down_u64(unsigned long long v, int d) {
    return __shfl_down_sync(0xffffffffu, v, d);
}
__device__ __forceinline__ double shfl_down_f64(double v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }

__device__ __forceinline__ void noise_shfl_down(NoiseAcc& r, const NoiseAcc& a, int d) {
    r.nrec = shfl_down_u32(a.nrec, d);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        r.b[i].s_b_fw = shfl_down_u64(a.b[i].s_b_fw, d); r.b[i].s_b_bw = shfl_down_u64(a.b[i].s_b_bw, d);
        r.b[i].s_d_fw = shfl_down_u64(a.b[i].s_d_fw, d); r.b[i].s_d_bw = shfl_down_u64(a.b[i].s_d_bw, d);
        r.b[i].s_p_fw = shfl_down_f64(a.b[i].s_p_fw, d); r.b[i].s_p_bw = shfl_down_f64(a.b[i].s_p_bw, d);
        r.b[i].count = shfl_down_u32(a.b[i].count, d);
        r.b[i].g_n = shfl_down_u32(a.b[i].g_n, d);
        r.b[i].g_first_x = shfl_down_u32(a.b[i].g_first_x, d); r.b[i].g_first_rd = shfl_down_u32(a.b[i].g_first_rd, d);
        r.b[i].g_x = shfl_down_u32(a.b[i].g_x, d); r.b[i].g_rd = shfl_down_u32(a.b[i].g_rd, d);
    }
}

// One warp per group.  Lane l takes the contiguous sample range [l*per, (l+1)*per); the partial states
// are merged in lane order by an order-preserving tree, which keeps the Germ_Max "first qualifying
// record is dropped" semantics (EE:1258-1262) exact.
__global__ void __launch_bounds__(128)
noise_twin_kernel(const uint4* __restrict__ counts, int S, int64_t P, const int32_t* __restrict__ twin_next,
                  const int32_t* __restrict__ heads, const uint32_t* __restrict__ counters, float C, uint32_t cut,
                  float* __restrict__ thr, float* __restrict__ germ_val, uint8_t* __restrict__ germ_state,
                  uint32_t* __restrict__ count, uint32_t* __restrict__ nrec) {
    const int lane = threadIdx.x & 31;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t n = counters[1];
    const int per = (S + 31) / 32;
    const int64_t sstride = 2 * P;
    for (uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < n; g += warps) {
        const int32_t head = heads[g];
        NoiseAcc acc;
        noise_init(acc);
        const int s_lo = lane * per, s_hi = min(S, s_lo + per);
        for (int s = s_lo; s < s_hi; ++s) {
            for (int32_t t = head; t >= 0; t = twin_next[t]) {  // rows of one file: slot order = file order
                const uint4 fw = ld_stream(counts + (int64_t)s * sstride + t);
                const uint4 bw = ld_stream(counts + (int64_t)s * sstride + P + t);
                noise_accumulate<true>(acc, fw, bw, C, cut);
            }
        }
#pragma unroll 1
        for (int d = 1; d < 32; d <<= 1) {
            NoiseAcc other;
            noise_shfl_down(other, acc, d);
            if ((lane & (2 * d - 1)) == 0) noise_merge(acc, other);
        }
        if (lane == 0)
            for (int32_t t = head; t >= 0; t = twin_next[t]) noise_store(acc, t, thr, germ_val, germ_state, count, nrec);
    }
}

// ------------------------------------------------------------------------------------------------
// uint16 wire format -> uint32 count words (the _host16 entry points): one thread per (sample, strand, slot) word
// ------------------------------------------------------------------------------------------------
__global__ void widen16_kernel(const uint2* __restrict__ in, uint4* __restrict__ out, int64_t n_words) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words) return;
    const uint2 v = in[i];
    uint4 o;
    if (v.x == 0xFFFFFFFFu && v.y == 0xFFFFFFFFu) {
        o = make_uint4(AS_ABSENT, AS_ABSENT, AS_ABSENT, AS_ABSENT);
    } else {
        o = make_uint4(v.x & 0xFFFFu, v.x >> 16, v.y & 0xFFFFu, v.y >> 16);
    }
    out[i] = o;
}

// packed wire format (include/amplisolve_b200.h): one word per (sample, strand, slot) = 16-bit major count, its base
// index, three 4-bit minor counts in ascending base order.  Escaped words become absent until patch_wide_kernel
// overwrites them with the record from the side list.
__global__ void unpack_kernel(const uint32_t* __restrict__ in, uint4* __restrict__ out, int64_t n_words) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words) return;
    const uint32_t w = in[i];
    uint4 o;
    if (w >= AS_PACKED_ESCAPE) {
        o = make_uint4(AS_ABSENT, AS_ABSENT, AS_ABSENT, AS_ABSENT);
    } else {
        const uint32_t m = w & 0xFFFFu, j = (w >> 16) & 3u;
        const uint32_t a = (w >> 18) & 15u, b = (w >> 22) & 15u, c = (w >> 26) & 15u;
        o.x = j == 0 ? m : a;
        o.y = j == 1 ? m : (j == 0 ? a : b);
        o.z = j == 2 ? m : (j == 3 ? c : b);
        o.w = j == 3 ? m : c;
    }
    out[i] = o;
}

// records whose counts do not fit 16 bits travel as as_wide_record; overwrite their (escaped) words in the tile
__global__ void patch_wide_kernel(const as_wide_record* __restrict__ wide, int64_t m, uint4* __restrict__ tile, int64_t n,
                                  int64_t p0, int n_samples) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const as_wide_record r = wide[i];
    const int64_t slot = (int64_t)r.slot - p0;
    if (slot < 0 || slot >= n || r.sample < 0 || r.sample >= n_samples) return;
    tile[((int64_t)r.sample * 2 + 0) * n + slot] = make_uint4(r.fw[0], r.fw[1], r.fw[2], r.fw[3]);
    tile[((int64_t)r.sample * 2 + 1) * n + slot] = make_uint4(r.bw[0], r.bw[1], r.bw[2], r.bw[3]);
}

// ------------------------------------------------------------------------------------------------
// thresholds as the caller sees them (EE:1787 "%f" text -> VC:889-890 std::stof)
// ------------------------------------------------------------------------------------------------
// four values per thread: the fp64 divide of thr_caller_view is a long dependent chain, four of them interleave
__global__ void thr_view_kernel(const float* __restrict__ thr, float* __restrict__ view, int64_t n) {
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i + 3 < n && ((reinterpret_cast<uintptr_t>(thr) | reinterpret_cast<uintptr_t>(view)) & 15) == 0) {
        const float4 v = *reinterpret_cast<const float4*>(thr + i);
        *reinterpret_cast<float4*>(view + i) = make_float4(thr_caller_view(v.x), thr_caller_view(v.y), thr_caller_view(v.z), thr_caller_view(v.w));
    } else {
        for (int64_t k = i; k < n && k < i + 4; ++k) view[k] = thr_caller_view(thr[k]);
    }
}

// ------------------------------------------------------------------------------------------------
// caller
// ------------------------------------------------------------------------------------------------
struct CallSlotConst {
    float e[8];    // thresholds of the slot as the caller parsed them: [base][fw,bw]
    uint32_t ref;  // 0..3, > 3 = not callable (VC:3290-3293)
};

__device__ __forceinline__ void load_slot_const(CallSlotConst& c, const float* __restrict__ thr_view,
                                                const uint8_t* __restrict__ ref, int64_t p) {
    const float4 a = *reinterpret_cast<const float4*>(thr_view + p * 8);
    const float4 b = *reinterpret_cast<const float4*>(thr_view + p * 8 + 4);
    c.e[0] = a.x; c.e[1] = a.y; c.e[2] = a.z; c.e[3] = a.w;
    c.e[4] = b.x; c.e[5] = b.y; c.e[6] = b.z; c.e[7] = b.w;
    c.ref = ref[p];
}

__device__ __forceinline__ void emit_call(as_call* __restrict__ calls, unsigned long long* __restrict__ n_calls,
                                          int64_t cap, bool is_call, int32_t sample, int32_t slot, int32_t alt,
                                          int32_t ref, double p_fw, double p_bw) {
    const unsigned active = __activemask();
    const unsigned votes = __ballot_sync(active, is_call);
    if (votes == 0) return;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(votes) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(n_calls, (unsigned long long)__popc(votes));
    base = __shfl_sync(active, base, leader);
    if (is_call) {
        const unsigned long long idx = base + __popc(votes & ((1u << lane) - 1u));
        if ((int64_t)idx < cap) {
            as_call c;
            c.sample = sample; c.slot = slot; c.alt = alt; c.ref = ref;
            c.p_fw = p_fw; c.p_bw = p_bw;
            c.q_fw = q_from_p(p_fw); c.q_bw = q_from_p(p_bw);
            calls[idx] = c;
        }
    }
}

// Straightforward version: one thread per (slot, sample chunk), strand tests evaluated in place.
// Kept as the in-tree cross-check of the queued kernel (tests compare both with the oracle).
__global__ void __launch_bounds__(AS_CALL_THREADS)
call_naive_kernel(const uint4* __restrict__ counts, int T, int64_t P, int64_t p0, int64_t p1, int chunk,
                  const uint8_t* __restrict__ ref, const float* __restrict__ thr_view, uint32_t cut,
                  as_call* __restrict__ calls, int64_t cap, unsigned long long* __restrict__ n_calls) {
    const int64_t p = p0 + (int64_t)blockIdx.x * AS_CALL_THREADS + threadIdx.x;
    if (p >= p1) return;
    CallSlotConst sc;
    load_slot_const(sc, thr_view, ref, p);
    if (sc.ref > 3) return;
    const int t0 = blockIdx.y * chunk, t1 = min(T, t0 + chunk);
    const int64_t sstride = 2 * P;
    for (int t = t0; t < t1; ++t) {
        const uint4 fw = ld_stream(counts + (int64_t)t * sstride + p);
        const uint4 bw = ld_stream(counts + (int64_t)t * sstride + P + p);
        if ((int32_t)fw.x < 0) continue;
        const uint32_t FW = fw.x + fw.y + fw.z + fw.w, BW = bw.x + bw.y + bw.z + bw.w;  // VC:760-770
        if (!(FW >= cut && BW >= cut)) continue;                                        // VC:898
        for (int b = 0; b < 4; ++b) {  // increasing base order = the alt order of VC:869-3288
            if ((uint32_t)b == sc.ref) continue;
            const uint32_t kf = comp(fw, b), kb = comp(bw, b);
            const float ef = sc.e[2 * b], eb = sc.e[2 * b + 1];
            bool is_call = false;
            double pf = 1.0, pb = 1.0;
            if (ef != -1.0f && eb != -1.0f) {
                pf = poisson_p((int)kf, (int)FW, ef);  // VC:895
                if (q_at_least_5(pf)) {
                    pb = poisson_p((int)kb, (int)BW, eb);  // VC:896
                    is_call = q_at_least_5(pb);
                }
            }
            emit_call(calls, n_calls, cap, is_call, t, (int32_t)p, b, (int32_t)sc.ref, pf, pb);
        }
    }
}

// Queued version.  Stage 0 (the scan): integer-only test per record and base -- coverage gate, alt != ref,
// alt reads > 0 on both strands (VC:3858-3861: k == 0 gives Q = 0).  Stage 1: candidates are compacted
// into a per-warp queue; full warps apply the exact m >= k screen.  Stage 2: survivors are compacted
// again and each takes TWO lanes (forward and reverse strand) for the fp64 series of VC:3785-3794.
struct CallCand {
    uint32_t k_fw, d_fw, k_bw, d_bw;
    float e_fw, e_bw;
    uint32_t sample_alt;  // sample | alt << 30
    int32_t slot;
};
static_assert(sizeof(CallCand) == 32, "CallCand is two 16-byte words");

#define AS_Q1_CAP 128 /* <= 31 left over + 32 lanes x 3 alts */
#define AS_Q2_CAP 48  /* <= 15 left over + 32 */

__device__ __forceinline__ void stage2_batch(const CallCand* __restrict__ q2, int n_pairs,
                                             const uint8_t* __restrict__ ref, as_call* __restrict__ calls,
                                             int64_t cap, unsigned long long* __restrict__ n_calls) {
    const int lane = threadIdx.x & 31;
    const int pair = lane >> 1, strand = lane & 1;
    double p = 1.0;
    CallCand c;
    const bool have = pair < n_pairs;
    if (have) {
        c = q2[pair];
        p = strand == 0 ? poisson_p((int)c.k_fw, (int)c.d_fw, c.e_fw) : poisson_p((int)c.k_bw, (int)c.d_bw, c.e_bw);
    }
    const double p_other = __shfl_xor_sync(0xffffffffu, p, 1);
    const bool is_call = have && strand == 0 && q_at_least_5(p) && q_at_least_5(p_other);
    const unsigned votes = __ballot_sync(0xffffffffu, is_call);
    if (votes == 0) return;
    const int leader = __ffs(votes) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(n_calls, (unsigned long long)__popc(votes));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (is_call) {
        const unsigned long long idx = base + __popc(votes & ((1u << lane) - 1u));
        if ((int64_t)idx < cap) {
            as_call o;
            o.sample = (int32_t)(c.sample_alt & 0x3fffffffu);
            o.slot = c.slot;
            o.alt = (int32_t)(c.sample_alt >> 30);
            o.ref = ref[c.slot];
            o.p_fw = p; o.p_bw = p_other;
            o.q_fw = q_from_p(p); o.q_bw = q_from_p(p_other);
            calls[idx] = o;
        }
    }
}

__device__ __forceinline__ void stage1_batch(const CallCand* __restrict__ q1, int n, CallCand* __restrict__ q2,
                                             int& n2, const uint8_t* __restrict__ ref, as_call* __restrict__ calls,
                                             int64_t cap, unsigned long long* __restrict__ n_calls) {
    const int lane = threadIdx.x & 31;
    CallCand c;
    bool surv = false;
    if (lane < n) {
        c = q1[lane];
        surv = strand_can_pass(c.k_fw, c.d_fw, c.e_fw) && strand_can_pass(c.k_bw, c.d_bw, c.e_bw);
    }
    const unsigned votes = __ballot_sync(0xffffffffu, surv);
    if (surv) q2[n2 + __popc(votes & ((1u << lane) - 1u))] = c;
    n2 += __popc(votes);
    __syncwarp();
    while (n2 >= 16) {
        stage2_batch(q2 + (n2 - 16), 16, ref, calls, cap, n_calls);
        n2 -= 16;
        __syncwarp();
    }
}

__global__ void __launch_bounds__(AS_CALL_THREADS)
call_queued_kernel(const uint4* __restrict__ counts, int T, int64_t P, int64_t p0, int64_t p1, int chunk,
                   const uint8_t* __restrict__ ref, const float* __restrict__ thr_view, uint32_t cut,
                   as_call* __restrict__ calls, int64_t cap, unsigned long long* __restrict__ n_calls) {
    __shared__ __align__(16) CallCand q1_all[AS_CALL_THREADS / 32][AS_Q1_CAP];
    __shared__ __align__(16) CallCand q2_all[AS_CALL_THREADS / 32][AS_Q2_CAP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    CallCand* q1 = q1_all[warp];
    CallCand* q2 = q2_all[warp];
    int n1 = 0, n2 = 0;  // warp-uniform

    const int64_t p = p0 + (int64_t)blockIdx.x * AS_CALL_THREADS + threadIdx.x;
    CallSlotConst sc;
    sc.ref = 255;
    if (p < p1) load_slot_const(sc, thr_view, ref, p);
    const bool slot_ok = p < p1 && sc.ref <= 3;
    // a warp whose lanes are all idle has nothing to scan (its queues stay empty)
    if (__ballot_sync(0xffffffffu, slot_ok) == 0) return;
    const int64_t pp = slot_ok ? p : p0;  // idle lanes read a valid address and discard it
    const uint32_t notref = slot_ok ? (0xfu & ~(1u << sc.ref)) : 0u;
    const int t0 = blockIdx.y * chunk, t1 = min(T, t0 + chunk);
    const int64_t sstride = 2 * P;

    for (int t = t0; t < t1; ++t) {
        const uint4 fw = ld_stream(counts + (int64_t)t * sstride + pp);
        const uint4 bw = ld_stream(counts + (int64_t)t * sstride + P + pp);
        const uint32_t FW = fw.x + fw.y + fw.z + fw.w, BW = bw.x + bw.y + bw.z + bw.w;
        uint32_t mask = 0;
        if ((int32_t)fw.x >= 0 && FW >= cut && BW >= cut) {
            mask = ((fw.x != 0 && bw.x != 0) ? 1u : 0u) | ((fw.y != 0 && bw.y != 0) ? 2u : 0u) |
                   ((fw.z != 0 && bw.z != 0) ? 4u : 0u) | ((fw.w != 0 && bw.w != 0) ? 8u : 0u);
            mask &= notref;
        }
        if (__ballot_sync(0xffffffffu, mask != 0) == 0) continue;
        // exclusive prefix sum of popc(mask) over the lanes
        const int mine = __popc(mask);
        int incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += up;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        int off = n1 + incl - mine;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            if (mask & (1u << b)) {
                CallCand c;
                c.k_fw = comp(fw, b); c.d_fw = FW; c.k_bw = comp(bw, b); c.d_bw = BW;
                c.e_fw = sc.e[2 * b]; c.e_bw = sc.e[2 * b + 1];
                c.sample_alt = (uint32_t)t | ((uint32_t)b << 30);
                c.slot = (int32_t)p;
                q1[off++] = c;
            }
        }
        n1 += total;
        __syncwarp();
        while (n1 >= 32) {
            stage1_batch(q1 + (n1 - 32), 32, q2, n2, ref, calls, cap, n_calls);
            n1 -= 32;
        }
    }
    if (n1 > 0) stage1_batch(q1, n1, q2, n2, ref, calls, cap, n_calls);
    if (n2 > 0) stage2_batch(q2, n2, ref, calls, cap, n_calls);
}

// n_c threshold tables (noise-floor sweep), c_stride floats apart; table ci owns the list calls + ci * cap and the
// counter n_calls[ci].  n_c == 1 is the plain caller.
__device__ __forceinline__ void stage2_batch_staged(const StagedCand* __restrict__ q2, int n_pairs,
                                                    const uint8_t* __restrict__ ref, const float* __restrict__ thr_view,
                                                    int n_c, int64_t c_stride, as_call* __restrict__ calls, int64_t cap,
                                                    unsigned long long* __restrict__ n_calls) {
    const int lane = threadIdx.x & 31;
    const int pair = lane >> 1, strand = lane & 1;
    double p = 1.0;
    StagedCand c;
    int ci = 0;
    const bool have = pair < n_pairs;
    if (have) {
        c = q2[pair];
        ci = (int)((c.sample_alt >> 27) & 7u);
        const float e = thr_view[(int64_t)ci * c_stride + (int64_t)c.slot * 8 + 2 * (c.sample_alt >> 30) + strand];
        p = strand == 0 ? poisson_p((int)c.k_fw, (int)c.d_fw, e) : poisson_p((int)c.k_bw, (int)c.d_bw, e);
    }
    const double p_other = __shfl_xor_sync(0xffffffffu, p, 1);
    const bool is_call = have && strand == 0 && q_at_least_5(p) && q_at_least_5(p_other);
    const unsigned votes = __ballot_sync(0xffffffffu, is_call);
    if (votes == 0) return;
    unsigned long long idx;
    if (n_c == 1) {  // one list: one atomic per batch
        const int leader = __ffs(votes) - 1;
        unsigned long long base = 0;
        if (lane == leader) base = atomicAdd(n_calls, (unsigned long long)__popc(votes));
        base = __shfl_sync(0xffffffffu, base, leader);
        idx = base + __popc(votes & ((1u << lane) - 1u));
    } else {         // one list per threshold table; calls are rare enough for one atomic each
        idx = is_call ? atomicAdd(n_calls + ci, 1ull) : 0ull;
        calls += (int64_t)ci * cap;
    }
    if (is_call) {
        if ((int64_t)idx < cap) {
            as_call o;
            o.sample = (int32_t)(c.sample_alt & 0x7ffffffu);
            o.slot = c.slot;
            o.alt = (int32_t)(c.sample_alt >> 30);
            o.ref = ref[c.slot];
            o.p_fw = p; o.p_bw = p_other;
            o.q_fw = q_from_p(p); o.q_bw = q_from_p(p_other);
            calls[idx] = o;
        }
    }
}

// TMA-staged caller.  Per stage every consumer thread scans its K records out of shared memory with integer
// tests only and keeps a 4-bit candidate mask per record; ONE warp prefix sum per stage compacts the
// candidates into 16-bit (record, lane, base) entries.  Full warps then revisit the candidates in the still
// resident stage for the exact m >= k screen; survivors go to the per-warp queue of fp64 series evaluations
// (two lanes per candidate, as in call_queued_kernel).
//
// PRE (integer pre-screen in the scan): the thread keeps, for its slot and each strand, R = floor(e_min * 2^32) of the
// SMALLEST threshold among the callable alt bases (and among the tables of a sweep).  prescreen_k turns the strand depth
// into a bound K: a strand test with 1 <= k <= K cannot reach Q >= 5 whatever the base, because its mean
// m = rn(depth * e_b) >= depth * e_min lies above the critical mean of strand_can_pass (or on the continued-fraction
// branch).  Such (record, base) pairs are dropped in the scan -- the "alt reads > 0" test k > 0 simply becomes k > K, at
// the price of one multiply per strand -- and never become candidates; pairs between K and their own base's bound still
// do and meet the exact fp64 screens in the revisit, so the call set is unchanged.  The candidate rate falls from 3 % (c3)
// / 15 % (c5 shape) of the pairs by one to two orders of magnitude.
// SWEEP: n_c_arg threshold tables, c_stride floats apart (noise-floor sweep: the tumour tensor is read once for all of
// them); otherwise one table and the loops over tables fold away.
template <int K, int STAGES, bool PRE, bool SWEEP>
__global__ void __launch_bounds__(AS_CTA_THREADS, SWEEP ? 6 : (PRE ? 7 : 1))
call_staged_kernel(const uint4* __restrict__ counts, int T, int64_t P, int64_t p0, int64_t p1, int chunk,
                   const uint8_t* __restrict__ ref, const float* __restrict__ thr_view, int n_c_arg, int64_t c_stride,
                   uint32_t cut, as_call* __restrict__ calls, int64_t cap, unsigned long long* __restrict__ n_calls) {
    const int n_c = SWEEP ? n_c_arg : 1;
    static_assert(K * 4 <= 32, "candidate mask is one 32-bit word per thread and stage");
    constexpr int CAND_CAP = K * 32 * 3;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * STAGES];
    __shared__ uint16_t cand_all[AS_CONSUMER_WARPS][CAND_CAP];
    __shared__ __align__(8) StagedCand q2_all[AS_CONSUMER_WARPS][AS_Q2_CAP];
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
    uint32_t Rf = 0, Rb = 0;  // PRE: floor(e_min * 2^32) per strand; 0 never screens anything out
    if (tid < n_slots) {
        const uint32_t r = ref[p];
        if (r <= 3) notref = 0xfu & ~(1u << r);
        if (PRE && r <= 3) {
            Rf = Rb = 0xFFFFFFFFu;
            for (int ci = 0; ci < n_c; ++ci) {  // the smallest threshold over the alt bases and over the tables of a sweep
            const float4 a = *reinterpret_cast<const float4*>(thr_view + ci * c_stride + p * 8);
            const float4 b = *reinterpret_cast<const float4*>(thr_view + ci * c_stride + p * 8 + 4);
            const float e[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if ((uint32_t)i == r) continue;
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    const float raw = e[2 * i + s];
                    if (raw == -1.0f) continue;  // no threshold: never a call (VC:3844-3849), puts no bound on the minimum
                    const float ee = effective_err(raw);
                    // e * 2^32 is exact (power-of-two scaling) and < 2^32 for e < 1; anything else (negative, NaN,
                    // e >= 1) switches the pre-screen off for the strand: the exact test decides
                    const uint32_t R = (ee > 0.0f && ee < 1.0f) ? __float2uint_rz(ee * 4294967296.0f) : 0u;
                    if (s == 0) Rf = min(Rf, R); else Rb = min(Rb, R);
                }
            }
            }
        }
    }
    uint16_t* cand = cand_all[warp];
    StagedCand* q2 = q2_all[warp];
    int n2 = 0;
    uint32_t notref_rep = notref;  // the 4-bit mask replicated for every record of a stage
#pragma unroll
    for (int j = 1; j < K; ++j) notref_rep |= notref << (4 * j);

    int it = 0;
    for (int t = t0; t < t1; t += K, ++it) {
        const uint4* st = ring.consumer_wait(it);
        const int k = min(K, t1 - t);
        // ---- scan: integer tests only (coverage gate VC:898, k == 0 -> Q = 0 VC:3858-3861, alt != ref)
        uint32_t mask = 0;
#pragma unroll
        for (int j = 0; j < K; ++j) {
            if (j < k) {
                const uint4 fw = st[(j * 2 + 0) * AS_TILE_SLOTS + tid];
                const uint4 bw = st[(j * 2 + 1) * AS_TILE_SLOTS + tid];
                const uint32_t FW = fw.x + fw.y + fw.z + fw.w, BW = bw.x + bw.y + bw.z + bw.w;
                uint32_t m;
                if (PRE) {
                    // a strand test with k <= K(m_lo) cannot pass; K = 0 leaves the plain k > 0 test
                    const uint32_t mf = prescreen_k(FW, Rf), mb = prescreen_k(BW, Rb);
                    m = ((fw.x > mf && bw.x > mb) ? 1u : 0u) | ((fw.y > mf && bw.y > mb) ? 2u : 0u) |
                        ((fw.z > mf && bw.z > mb) ? 4u : 0u) | ((fw.w > mf && bw.w > mb) ? 8u : 0u);
                } else {
                    m = ((min(fw.x, bw.x) != 0) ? 1u : 0u) | ((min(fw.y, bw.y) != 0) ? 2u : 0u) |
                        ((min(fw.z, bw.z) != 0) ? 4u : 0u) | ((min(fw.w, bw.w) != 0) ? 8u : 0u);
                }
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
            // ---- revisit the candidates with full warps: exact m >= k screen, survivors to the series queue
            for (int base = 0; base < total; base += 32) {
                const int i = base + lane;
                uint4 w0 = make_uint4(0, 0, 0, 0);  // the StagedCand as a 16-byte and an 8-byte word
                uint2 w1 = make_uint2(0, 0);
                const float* ethr = thr_view;       // thresholds of the candidate's (slot, base): a rare read, served by L2
                if (i < total) {
                    const uint32_t e = cand[i];
                    const int src = e & 31, bit = e >> 5, j = bit >> 2, b = bit & 3;
                    const int col = warp * 32 + src;
                    const uint4 fw = st[(j * 2 + 0) * AS_TILE_SLOTS + col];
                    const uint4 bw = st[(j * 2 + 1) * AS_TILE_SLOTS + col];
                    ethr = thr_view + (tile0 + col) * 8 + 2 * b;
                    w0 = make_uint4(comp(fw, b), fw.x + fw.y + fw.z + fw.w, comp(bw, b), bw.x + bw.y + bw.z + bw.w);
                    w1 = make_uint2((uint32_t)(t + j) | ((uint32_t)b << 30), (uint32_t)(tile0 + col));
                }
                // one exact screen per threshold table of a sweep; the threshold reads of all tables are issued together
                // (independent L2 reads), the queue pushes follow table by table
                uint32_t smask = 0;
                if (i < total) {
                    if (SWEEP) {
#pragma unroll
                        for (int ci = 0; ci < 8; ++ci) {
                            if (ci < n_c) {
                                const float2 ee = *reinterpret_cast<const float2*>(ethr + ci * c_stride);
                                smask |= (strand_can_pass(w0.x, w0.y, ee.x) && strand_can_pass(w0.z, w0.w, ee.y)) ? (1u << ci) : 0u;
                            }
                        }
                    } else {
                        const float2 ee = *reinterpret_cast<const float2*>(ethr);
                        smask = (strand_can_pass(w0.x, w0.y, ee.x) && strand_can_pass(w0.z, w0.w, ee.y)) ? 1u : 0u;
                    }
                }
                if (SWEEP && __ballot_sync(0xffffffffu, smask != 0) == 0) continue;
                for (int ci = 0; ci < n_c; ++ci) {
                    const bool surv = (smask >> ci) & 1u;
                    const unsigned votes = __ballot_sync(0xffffffffu, surv);
                    if (surv) {
                        uint2* dst = reinterpret_cast<uint2*>(q2 + n2 + __popc(votes & ((1u << lane) - 1u)));
                        dst[0] = make_uint2(w0.x, w0.y);
                        dst[1] = make_uint2(w0.z, w0.w);
                        dst[2] = make_uint2(w1.x | ((uint32_t)ci << 27), w1.y);
                    }
                    n2 += __popc(votes);
                    __syncwarp();
                    while (n2 >= 16) {
                        stage2_batch_staged(q2 + (n2 - 16), 16, ref, thr_view, n_c, c_stride, calls, cap, n_calls);
                        n2 -= 16;
                        __syncwarp();
                    }
                }
            }
        }
        ring.consumer_release(it);
    }
    if (n2 > 0) stage2_batch_staged(q2, n2, ref, thr_view, n_c, c_stride, calls, cap, n_calls);
}

// Forward-first caller.  A record can only become a call if BOTH strand tests pass (VC:898, VC:895-896), and the forward
// strand alone rules out nearly every record: the ring streams the forward plane only (16 B per record instead of 32).
// The CTA's warps have two roles: four scan warps and one control warp per ring stage.
// Scan warps (warps 0-3, thread per slot), every record, integer only and branch-free: present, FW >= cut, and
// k > prescreen_k(FW, R_min) for some callable base (alt != ref, a threshold on both strands: -1 is never a call,
// VC:3844-3849), R_min = floor(e * 2^32) of the smallest forward threshold of those bases.  A thread stores one K-bit pass
// mask per stage and releases the stage; the arrive on the stage's empty barrier publishes the mask.
// Control warp c (warp 4 + c) owns stage c.  Each time the scan warps have released it (it is the stage's last reader):
//   1. the 128 pass masks, one warp prefix sum -> the list of passing (record, column);
//   2. 32 passers at a time, one per lane: each base against its own bound R_b (what the bound of strand_can_pass is; the
//      minimum is only weaker, and one multiply per record is what keeps the scan lean);
//   3. the records with a candidate base, compacted by ballot into the warp's pending ring: the forward word, (sample,
//      column | base mask), and the reverse-strand word, fetched with a 16-byte cp.async; one commit group per stage;
//   4. the refill of the stage (bulk copies of the forward rows);
//   5. then, off the refill path, the pending entries of the warp's stage i are resolved at its stage i + D or later, once
//      a warp's worth has landed: BW >= cut, reverse k > prescreen_k(BW, R_b), strand_can_pass on both strands; survivors join the series
//      queue of call_staged_kernel.
// The per-record candidate work is thus paid once per CTA and stage, on full warps, instead of in every scan warp.  It is
// still a chain of dependent shared-memory reads, shuffles and fp64 series on one warp; one control warp per stage lets the
// control work of consecutive stages overlap (one control warp for all stages was slower than the per-warp design it
// replaces, DESIGN 3.2b).  A ring that cannot take a stage's candidates is drained on the spot (wait for every copy,
// resolve), a slower path that gives the same calls; pend_cap < AS_FWD_PENDING caps the usable depth (tests of that path).
struct FwdPending {  // per control warp; the reverse words are cp.async targets (16-byte aligned)
    uint4 bw[AS_FWD_PENDING];
    uint4 fw[AS_FWD_PENDING];
    uint2 meta[AS_FWD_PENDING];  // sample, tile column | forward candidate base mask << 8
};

// resolve the n pending entries from ring entry `from` on; full warps, one entry per lane
__device__ __forceinline__ void fwd_resolve(const FwdPending& pd, uint32_t from, uint32_t n, const float (*thr_s)[8], int64_t tile0,
                                            uint32_t cut, StagedCand* __restrict__ q2, int& n2, const uint8_t* __restrict__ ref,
                                            const float* __restrict__ thr_view, as_call* __restrict__ calls, int64_t cap,
                                            unsigned long long* __restrict__ n_calls) {
    const int lane = threadIdx.x & 31;
    for (uint32_t base = 0; base < n; base += 32) {
        const uint32_t i = base + lane;
        const uint32_t pos = (from + i) & (AS_FWD_PENDING - 1);
        uint32_t smask = 0;
        if (i < n) {
            const uint4 fw = pd.fw[pos], bw = pd.bw[pos];
            const uint2 meta = pd.meta[pos];
            const uint32_t FW = fw.x + fw.y + fw.z + fw.w, BW = bw.x + bw.y + bw.z + bw.w;
            const uint32_t fm = meta.y >> 8;
            const float* e = thr_s[meta.y & 255u];
            if (BW >= cut) {
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    if ((fm >> b) & 1u) {
                        const uint32_t kb = comp(bw, b);
                        const float ee = effective_err(e[2 * b + 1]);
                        const uint32_t R = (ee > 0.0f && ee < 1.0f) ? __float2uint_rz(ee * 4294967296.0f) : 0u;
                        if (kb > prescreen_k(BW, R) && strand_can_pass(comp(fw, b), FW, e[2 * b]) && strand_can_pass(kb, BW, e[2 * b + 1]))
                            smask |= 1u << b;
                    }
                }
            }
        }
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const bool surv = (smask >> b) & 1u;
            const unsigned votes = __ballot_sync(0xffffffffu, surv);
            if (votes == 0) continue;
            if (surv) {  // the entry is read again from the ring: nothing of it stays live across the series below
                const uint4 fw = pd.fw[pos], bw = pd.bw[pos];
                const uint2 meta = pd.meta[pos];
                uint2* dst = reinterpret_cast<uint2*>(q2 + n2 + __popc(votes & ((1u << lane) - 1u)));
                dst[0] = make_uint2(comp(fw, b), fw.x + fw.y + fw.z + fw.w);
                dst[1] = make_uint2(comp(bw, b), bw.x + bw.y + bw.z + bw.w);
                dst[2] = make_uint2(meta.x | ((uint32_t)b << 30), (uint32_t)(tile0 + (meta.y & 255u)));
            }
            n2 += __popc(votes);
            __syncwarp();
            while (n2 >= 16) {
                stage2_batch_staged(q2 + (n2 - 16), 16, ref, thr_view, 1, 0, calls, cap, n_calls);
                n2 -= 16;
                __syncwarp();
            }
        }
    }
    __syncwarp();  // the entries are read before the ring positions are reused
}

// (4, 3): 224 threads, 4 CTAs/SM; registers (one allocation for both roles: 72 per thread, set by the control warps'
// fp64 series) and shared memory (24 KiB of stages + 28 KiB of tables and per-warp queues) both allow four, neither five.
template <int K, int STAGES, int D>
__global__ void __launch_bounds__(AS_TILE_SLOTS + 32 * STAGES, 4)
call_forward_kernel(const uint4* __restrict__ counts, int T, int64_t P, int64_t p0, int64_t p1, int chunk,
                    const uint8_t* __restrict__ ref, const float* __restrict__ thr_view, uint32_t cut, int pend_cap,
                    as_call* __restrict__ calls, int64_t cap, unsigned long long* __restrict__ n_calls) {
    static_assert(K <= 8, "a record's pass bit in one byte per slot and stage");
    static_assert(D >= 1 && D <= 4, "resolution distance in stages");
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * STAGES];
    __shared__ __align__(16) float thr_s[AS_TILE_SLOTS][8];
    __shared__ __align__(16) uint4 rb_s[AS_TILE_SLOTS];     // floor(e_b * 2^32) of the forward threshold of each base
    __shared__ uint32_t callable_s[AS_TILE_SLOTS];           // callable-base mask
    __shared__ __align__(4) uint8_t pass_s[STAGES][AS_TILE_SLOTS];  // scan -> control: bit j = record j of the stage passes
    __shared__ uint16_t passers_all[STAGES][K * AS_TILE_SLOTS];  // record << 8 | column, of the stage a control warp reads
    __shared__ __align__(16) FwdPending pd_all[STAGES];
    __shared__ __align__(8) StagedCand q2_all[STAGES][AS_Q2_CAP];
    const int64_t tile0 = p0 + (int64_t)blockIdx.x * AS_TILE_SLOTS;
    const int n_slots = (int)min((int64_t)AS_TILE_SLOTS, p1 - tile0);
    const int t0 = blockIdx.y * chunk, t1 = min(T, t0 + chunk);
    const int tid = threadIdx.x, lane = tid & 31;
    uint32_t Rmin = 0xFFFFFFFFu, callable = 0;
    if (tid < AS_TILE_SLOTS) {
        uint32_t Rf[4] = {0u, 0u, 0u, 0u};  // 0 screens nothing out
        const int64_t p = tile0 + tid;
        if (tid < n_slots) {
            const float4 a = *reinterpret_cast<const float4*>(thr_view + p * 8);
            const float4 b = *reinterpret_cast<const float4*>(thr_view + p * 8 + 4);
            *reinterpret_cast<float4*>(&thr_s[tid][0]) = a;
            *reinterpret_cast<float4*>(&thr_s[tid][4]) = b;
            const float e[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
            const uint32_t r = ref[p];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (r > 3 || (uint32_t)i == r || e[2 * i] == -1.0f || e[2 * i + 1] == -1.0f) continue;
                callable |= 1u << i;
                // e * 2^32 is exact (power-of-two scaling) and < 2^32 for e < 1; anything else (negative, NaN, e >= 1)
                // switches the pre-screen off for the base: the exact tests decide
                const float ee = effective_err(e[2 * i]);
                Rf[i] = (ee > 0.0f && ee < 1.0f) ? __float2uint_rz(ee * 4294967296.0f) : 0u;
                Rmin = min(Rmin, Rf[i]);
            }
        }
        rb_s[tid] = make_uint4(Rf[0], Rf[1], Rf[2], Rf[3]);
        callable_s[tid] = callable;
    }
    StageRing<K, STAGES, 1> ring;
    ring.init(smem_raw, bars);  // its __syncthreads also publishes the tables above to the control warps
    const int n_it = (t1 - t0 + K - 1) / K;

    if (tid < AS_TILE_SLOTS) {
        // ---- scan warps: present, FW >= cut, and one pre-screen bound against the smallest forward threshold of the
        // callable bases (k > K(R_min) for some callable base) -- one multiply per record.  A slot past the tile's end has
        // no callable base and never passes.
        const uint32_t ax = 0u - (callable & 1u), ay = 0u - ((callable >> 1) & 1u), az = 0u - ((callable >> 2) & 1u),
                       aw = 0u - (callable >> 3);
        for (int it = 0; it < n_it; ++it) {
            const uint4* st = ring.consumer_wait(it);
            const int k = min(K, t1 - t0 - it * K);
            uint32_t rec = 0;  // one bit per record that passes
#pragma unroll
            for (int j = 0; j < K; ++j) {  // records j >= k hold stale words: dropped below
                const uint4 fw = st[j * AS_TILE_SLOTS + tid];
                const uint32_t FW = fw.x + fw.y + fw.z + fw.w;
                const uint32_t kmax = max(max(fw.x & ax, fw.y & ay), max(fw.z & az, fw.w & aw));
                const bool pass = ((int32_t)fw.x >= 0) & (FW >= cut) & (kmax > prescreen_k(FW, Rmin));  // no branches
                rec |= pass ? (1u << j) : 0u;
            }
            pass_s[it % STAGES][tid] = (uint8_t)(rec & ((1u << k) - 1u));
            ring.consumer_release(it);
        }
        return;
    }

    // ---- control warps: warp c owns stage c (iterations c, c + STAGES, ...)
    const int cw = (tid - AS_TILE_SLOTS) >> 5;
    uint16_t* passers = passers_all[cw];
    FwdPending& pd = pd_all[cw];
    StagedCand* q2 = q2_all[cw];
    const uint4* src = counts + tile0;
    const int64_t sstride = 2 * P;
    const uint32_t row_bytes = (uint32_t)n_slots * 16u;
    if (lane == 0 && cw < n_it) ring.fill(cw, src, sstride, P, t0, t1, row_bytes);
    const uint4* bw_tile = counts + P + tile0;  // reverse word of (sample s, column c) at bw_tile + s * 2P + c
    const int cap_pend = (pend_cap > 0 && pend_cap < AS_FWD_PENDING) ? pend_cap : AS_FWD_PENDING;
    const int batch = min(cap_pend, 32);
    int n2 = 0;
    uint32_t head = 0, tail = 0;  // running entry counts; entries [tail, head) are pending (wrap-safe differences)
    uint32_t ends[D + 1];         // ends[d] = head after the stage d stages back
#pragma unroll
    for (int d = 0; d <= D; ++d) ends[d] = 0;

    for (int it = cw; it < n_it; it += STAGES) {
        const int s = cw;
        const uint32_t parity = (it / STAGES) & 1;
        mbar_wait(&ring.empty[s], parity);  // every scan warp has stored its pass masks and released the stage
        mbar_wait(&ring.full[s], parity);   // completed long ago; makes the visibility of the bulk-copied words explicit
        const uint4* st = ring.stage(s);
        const int t = t0 + it * K;
        // 1. the passers of the stage: four columns per lane, one prefix sum
        const uint32_t pm = reinterpret_cast<const uint32_t*>(pass_s[s])[lane];
        const int mine = __popc(pm);
        int incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += up;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        for (uint32_t m = pm, o = incl - mine; m != 0; m &= m - 1, ++o) {
            const int bit = __ffs(m) - 1;
            passers[o] = (uint16_t)(((bit & 7) << 8) | (lane * 4 + (bit >> 3)));
        }
        __syncwarp();
        // 2.-3. each passer's bases against their own bounds; the candidates into the pending ring
        for (int base = 0; base < total; base += 32) {
            const int i = base + lane;
            uint4 fw = make_uint4(0, 0, 0, 0);
            uint32_t bm = 0, j = 0, col = 0;
            if (i < total) {
                const uint32_t e = passers[i];
                j = e >> 8;
                col = e & 255u;
                fw = st[j * AS_TILE_SLOTS + col];
                const uint4 Rf = rb_s[col];
                const uint32_t FW = fw.x + fw.y + fw.z + fw.w;
                bm = ((fw.x > prescreen_k(FW, Rf.x) ? 1u : 0u) | (fw.y > prescreen_k(FW, Rf.y) ? 2u : 0u) |
                      (fw.z > prescreen_k(FW, Rf.z) ? 4u : 0u) | (fw.w > prescreen_k(FW, Rf.w) ? 8u : 0u)) & callable_s[col];
            }
            unsigned votes = __ballot_sync(0xffffffffu, bm != 0);
            while (votes != 0) {
                if ((int)(head - tail) == cap_pend) {  // the ring is full: drain it on the spot
                    cp_async_commit();
                    cp_async_wait<0>();
                    __syncwarp();
                    fwd_resolve(pd, tail, head - tail, thr_s, tile0, cut, q2, n2, ref, thr_view, calls, cap, n_calls);
                    tail = head;
                }
                const uint32_t room = (uint32_t)cap_pend - (head - tail);
                const uint32_t rank = __popc(votes & ((1u << lane) - 1u));
                const bool take = ((votes >> lane) & 1u) && rank < room;
                if (take) {
                    const uint32_t pos = (head + rank) & (AS_FWD_PENDING - 1);
                    pd.fw[pos] = fw;
                    pd.meta[pos] = make_uint2((uint32_t)t + j, col | (bm << 8));
                    cp_async16(&pd.bw[pos], bw_tile + (int64_t)(t + (int)j) * sstride + col);
                }
                const unsigned taken = __ballot_sync(0xffffffffu, take);
                head += (uint32_t)__popc(taken);
                votes &= ~taken;
            }
        }
        cp_async_commit();
        // 4. the stage has been read for the last time: refill it
        __syncwarp();
        if (lane == 0 && it + STAGES < n_it) ring.fill(it + STAGES, src, sstride, P, t0, t1, row_bytes);
        // 5. entries of the stages D and more back have landed (every commit group but the D most recent); they are
        // resolved once there are enough of them to keep the warp's lanes busy, not every stage
#pragma unroll
        for (int d = D; d > 0; --d) ends[d] = ends[d - 1];
        ends[0] = head;
        if ((int)(ends[D] - tail) >= batch) {
            cp_async_wait<D>();
            __syncwarp();
            fwd_resolve(pd, tail, ends[D] - tail, thr_s, tile0, cut, q2, n2, ref, thr_view, calls, cap, n_calls);
            tail = ends[D];
        }
    }
    if (head != tail) {
        cp_async_wait<0>();
        __syncwarp();
        fwd_resolve(pd, tail, head - tail, thr_s, tile0, cut, q2, n2, ref, thr_view, calls, cap, n_calls);
    }
    if (n2 > 0) stage2_batch_staged(q2, n2, ref, thr_view, 1, 0, calls, cap, n_calls);
}

// ------------------------------------------------------------------------------------------------
// element-wise evaluators (parity grids)
// ------------------------------------------------------------------------------------------------
__global__ void poisson_test_kernel(const int32_t* __restrict__ k, const int32_t* __restrict__ rd,
                                    const float* __restrict__ err, int64_t n, double* __restrict__ p,
                                    double* __restrict__ q) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (err[i] == -1.0f) { p[i] = __longlong_as_double(0x7ff8000000000000ull); q[i] = -888.0; return; }  // VC:3844
    const double pv = poisson_p(k[i], rd[i], err[i]);
    p[i] = pv;
    q[i] = q_from_p(pv);
}

__global__ void gammaq_kernel(const double* __restrict__ s, const double* __restrict__ z, int64_t n,
                              double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = kf_gammaq(s[i], z[i]);
}

// ------------------------------------------------------------------------------------------------
// synthetic panels generated in HBM (SURVEY.md 8d); not on the parity path
// ------------------------------------------------------------------------------------------------
// Synthetic panel geometry: amplicons of AS_SYNTH_AMPLICON slots; one junction in `twin_period` (0 = none) overlaps
// the next amplicon by 2..10 positions, which then own two slots each (SURVEY.md 8d: ~1.6 % duplicated slots at
// period 6).  overlap(a) is the overlap of amplicon a with a+1; it is 0 when a+1 is not completely inside the shard.
#define AS_SYNTH_AMPLICON 125
__device__ __forceinline__ int synth_overlap(const as_synth_params& prm, int64_t a, int64_t P) {
    if (prm.twin_period <= 0 || a < 0) return 0;
    const int64_t first = prm.slot_offset / AS_SYNTH_AMPLICON;  // shards start on amplicon boundaries
    if ((a + 2 - first) * AS_SYNTH_AMPLICON > P || a < first) return 0;
    const uint64_t h = key4(prm.seed, (uint64_t)a, 0x50, 0);
    return (h % (uint64_t)prm.twin_period) == 0 ? 2 + (int)((h >> 20) % 9) : 0;
}
// first slot (global index) of the position that global slot g enumerates
__device__ __forceinline__ int64_t synth_head(const as_synth_params& prm, int64_t g, int64_t P) {
    const int64_t a = g / AS_SYNTH_AMPLICON, j = g % AS_SYNTH_AMPLICON;
    const int ov = synth_overlap(prm, a - 1, P);
    return j < ov ? (a - 1) * AS_SYNTH_AMPLICON + AS_SYNTH_AMPLICON - ov + j : g;
}

__global__ void synth_twin_links_kernel(int64_t P, as_synth_params prm, int32_t* __restrict__ twin_next,
                                        int32_t* __restrict__ twin_head) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const int64_t g = p + prm.slot_offset;
    const int64_t a = g / AS_SYNTH_AMPLICON, j = g % AS_SYNTH_AMPLICON;
    twin_head[p] = (int32_t)(synth_head(prm, g, P) - prm.slot_offset);
    const int ov = synth_overlap(prm, a, P);
    twin_next[p] = j >= AS_SYNTH_AMPLICON - ov ? (int32_t)((a + 1) * AS_SYNTH_AMPLICON + j - (AS_SYNTH_AMPLICON - ov) - prm.slot_offset)
                                               : -1;
}

__global__ void synth_kernel(uint4* __restrict__ counts, int n_samples, int64_t P, uint8_t* __restrict__ ref_out,
                             as_synth_params prm) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    // all randomness is keyed by the POSITION, so the slots of a duplicated position carry identical rows
    const uint64_t gp = (uint64_t)synth_head(prm, p + prm.slot_offset, P);
    const uint64_t hs = key4(prm.seed, gp, 0x51, 0);
    const uint32_t ref = (uint32_t)(hs & 3);
    if (ref_out != nullptr && blockIdx.y == 0) ref_out[p] = (uint8_t)ref;
    // per-amplicon depth multiplier, shared by all samples (125-slot amplicons)
    const float amp = __expf(0.6f * gauss(key4(prm.seed, gp / 125, 0x52, 0)));
    // per (slot, base, strand) error rate: 0 with probability 0.6, else log-normal around 3e-4, capped at 0.02
    float e[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint64_t h = key4(prm.seed, gp, 0x53, j);
        e[j] = (u01(h) < 0.6f) ? 0.0f : fminf(0.02f, 3e-4f * __expf(gauss(mix64(h))));
    }
    // germline SNP of the slot: alt base and which samples carry it (population frequency 0.2)
    const bool snp = u01(key4(prm.seed, gp, 0x54, 0)) < prm.germline_rate;
    const uint32_t snp_alt = (ref + 1 + (uint32_t)((hs >> 8) % 3)) & 3;

    const int s_per = (n_samples + gridDim.y - 1) / gridDim.y;
    const int s0 = blockIdx.y * s_per, s1 = min(n_samples, s0 + s_per);
    for (int s = s0; s < s1; ++s) {
        const uint64_t gs = (uint64_t)(s + prm.sample_offset);
        const uint64_t h = key4(prm.seed, gp, 0x60, gs);
        uint4 fw, bw;
        const float depth = prm.mean_depth * amp * __expf(prm.depth_sigma * gauss(h));
        if (u01(mix64(h ^ 0x1111)) < prm.absent_rate || depth < 20.0f) {
            fw = bw = make_uint4(AS_ABSENT, AS_ABSENT, AS_ABSENT, AS_ABSENT);
        } else {
            const float half = 0.5f * depth;
            const float dfw = fmaxf(0.0f, half + sqrtf(0.5f * half) * gauss(mix64(h ^ 0x2222)));
            const float dbw = fmaxf(0.0f, depth - dfw);
            float vaf[4] = {0.f, 0.f, 0.f, 0.f};  // true variant allele fractions on top of the noise
            if (snp && u01(key4(prm.seed, gp, 0x55, gs)) < 0.2f)
                vaf[snp_alt] = (key4(prm.seed, gp, 0x56, gs) & 1) ? 1.0f : 0.5f;
            const uint64_t hm = key4(prm.seed, gp, 0x57, gs);
            if (u01(hm) < prm.somatic_rate) {
                const uint32_t alt = (ref + 1 + (uint32_t)((hm >> 3) % 3)) & 3;
                vaf[alt] = fmaxf(vaf[alt], prm.somatic_vaf_lo + (prm.somatic_vaf_hi - prm.somatic_vaf_lo) * u01(mix64(hm)));
            }
            uint32_t c[8];
            uint32_t alt_fw = 0, alt_bw = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                if ((uint32_t)b == ref) { c[b] = c[4 + b] = 0; continue; }
                const float rf = fminf(1.0f, e[b] + vaf[b]), rb = fminf(1.0f, e[4 + b] + vaf[b]);
                c[b] = min(poisson_sample(dfw * rf, key4(prm.seed, gp, 0x70 + b, gs)), (uint32_t)dfw - alt_fw);
                c[4 + b] = min(poisson_sample(dbw * rb, key4(prm.seed, gp, 0x78 + b, gs)), (uint32_t)dbw - alt_bw);
                alt_fw += c[b]; alt_bw += c[4 + b];
            }
            c[ref] = (uint32_t)dfw - alt_fw;
            c[4 + ref] = (uint32_t)dbw - alt_bw;
            fw = make_uint4(c[0], c[1], c[2], c[3]);
            bw = make_uint4(c[4], c[5], c[6], c[7]);
        }
        counts[(int64_t)s * 2 * P + p] = fw;
        counts[(int64_t)s * 2 * P + P + p] = bw;
    }
}

}  // namespace asdev

// ================================================================================================
// launchers (plain C++ signatures, used by as_capi.cu)
// ================================================================================================
using namespace asdev;

static inline unsigned cdiv64(int64_t a, int64_t b) { return (unsigned)((a + b - 1) / b); }

template <int K, int STAGES>
static cudaError_t launch_noise_staged(const uint4* c, int S, int64_t P, int64_t p0, int64_t p1, const int32_t* tn,
                                       const int32_t* th, int64_t twin_base, float C, uint32_t cut, float* thr,
                                       float* gv, uint8_t* gs, uint32_t* cnt, uint32_t* nrec, cudaStream_t st) {
    static bool configured[AS_MAX_DEVICES] = {};  // the attribute is per device
    const int smem = StageRing<K, STAGES>::kStageBytes * STAGES;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= AS_MAX_DEVICES || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(noise_staged_kernel<K, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < AS_MAX_DEVICES) configured[dev] = true;
    }
    noise_staged_kernel<K, STAGES><<<cdiv64(p1 - p0, AS_TILE_SLOTS), AS_CTA_THREADS, smem, st>>>(
        c, S, P, p0, p1, tn, th, twin_base, C, cut, thr, gv, gs, cnt, nrec);
    return cudaGetLastError();
}

cudaError_t as_launch_noise_main(int cfg, const uint32_t* d_counts, int S, int64_t P, int64_t p0, int64_t p1,
                                 const int32_t* d_twin_next, const int32_t* d_twin_head, int64_t twin_base, float C,
                                 uint32_t cut, float* d_thr, float* d_germ_val, uint8_t* d_germ_state,
                                 uint32_t* d_count, uint32_t* d_nrec, cudaStream_t st) {
    if (p1 <= p0) return cudaSuccess;
    const uint4* c = reinterpret_cast<const uint4*>(d_counts);
#define AS_NOISE_ARGS c, S, P, p0, p1, d_twin_next, d_twin_head, twin_base, C, cut, d_thr, d_germ_val, d_germ_state, d_count, d_nrec
    if (cfg >= 7)  // register-lean pattern kernel (as_noise_pattern.cu), one value of C
        return as_launch_noise_pattern(cfg - 7, d_counts, S, P, p0, p1, d_twin_next, d_twin_head, twin_base, &C, 1, cut, d_thr, 0,
                                       d_germ_val, d_germ_state, d_count, d_nrec, st);
    switch (cfg) {
        case 0:
            noise_main_kernel<AS_NOISE_UNROLL><<<cdiv64(p1 - p0, AS_NOISE_THREADS), AS_NOISE_THREADS, 0, st>>>(AS_NOISE_ARGS);
            return cudaGetLastError();
        case 4: return launch_noise_staged<8, 2>(AS_NOISE_ARGS, st);
        case 6: return launch_noise_staged<4, 2>(AS_NOISE_ARGS, st);
        default: return launch_noise_staged<4, 3>(AS_NOISE_ARGS, st);
    }
#undef AS_NOISE_ARGS
}

// Twin groups the streaming kernel leaves out.  as_launch_twin_heads (memset + 1 kernel) lists them -- pairs in the first
// half of d_heads_scratch, longer groups in the second, d_counters two uint32 -- and as_launch_noise_twin_groups (2
// kernels) reduces them for one value of C.  cfg = the streaming kernel's variant (decides who owns in-tile pairs).
cudaError_t as_launch_twin_heads(int cfg, int64_t p0, int64_t p1, const int32_t* d_twin_next, const int32_t* d_twin_head,
                                 int32_t* d_heads_scratch, uint32_t* d_counters, cudaStream_t st) {
    if (p1 <= p0 || d_twin_next == nullptr) return cudaSuccess;
    const int64_t half = (p1 - p0 + 1) / 2 + 1;
    cudaMemsetAsync(d_counters, 0, 2 * sizeof(uint32_t), st);
    // in-tile pairs are reduced by the staged kernel when its ring can hold the hand-over block (see kPairsInTile)
    int ring_kb = 0;
    switch (cfg) { case 0: ring_kb = 0; break; case 4: ring_kb = 64; break; case 6: ring_kb = 32; break; default: ring_kb = 48; }
    // cfg >= 7: noise_pattern_kernel, which always merges in-tile pairs itself
    const int skip_intile = cfg >= 7 ? 1 : ((AS_INTILE_TWINS && ring_kb * 1024 >= AS_TILE_SLOTS * (int)sizeof(PairXfer)) ? 1 : 0);
    twin_heads_kernel<<<cdiv64(p1 - p0, 256), 256, 0, st>>>(d_twin_next, d_twin_head, p0, p1, skip_intile, d_heads_scratch,
                                                           d_heads_scratch + half, d_counters);
    return cudaGetLastError();
}

cudaError_t as_launch_noise_twin_groups(const uint32_t* d_counts, int S, int64_t P, int64_t p0, int64_t p1,
                                        const int32_t* d_twin_next, const int32_t* d_heads_scratch, const uint32_t* d_counters,
                                        float C, uint32_t cut, float* d_thr, float* d_germ_val, uint8_t* d_germ_state,
                                        uint32_t* d_count, uint32_t* d_nrec, cudaStream_t st) {
    if (p1 <= p0 || d_twin_next == nullptr) return cudaSuccess;
    const uint4* c = reinterpret_cast<const uint4*>(d_counts);
    const int64_t half = (p1 - p0 + 1) / 2 + 1;
    // pairs: at most (p1-p0)/2 quads; enough CTAs to cover a typical panel (~1 % of the slots) in one pass
    const unsigned pair_grid = (unsigned)std::min<int64_t>(148 * 16, std::max<int64_t>(1, (p1 - p0) / 64 / 32 + 1));  // 32 pairs per CTA
    noise_pair_kernel<<<pair_grid, 128, 0, st>>>(c, S, P, d_twin_next, d_heads_scratch, d_counters, C, cut, d_thr, d_germ_val,
                                                 d_germ_state, d_count, d_nrec);
    const unsigned grid = (unsigned)std::min<int64_t>(148 * 2, std::max<int64_t>(1, (p1 - p0 + 7) / 8));
    noise_twin_kernel<<<grid, 128, 0, st>>>(c, S, P, d_twin_next, d_heads_scratch + half, d_counters, C, cut, d_thr, d_germ_val,
                                            d_germ_state, d_count, d_nrec);
    return cudaGetLastError();
}

// 4 launches (memset node + 3 kernels): heads, then the groups for one value of C
cudaError_t as_launch_noise_twins(int cfg, const uint32_t* d_counts, int S, int64_t P, int64_t p0, int64_t p1,
                                  const int32_t* d_twin_next, const int32_t* d_twin_head, int32_t* d_heads_scratch,
                                  uint32_t* d_counters, float C, uint32_t cut, float* d_thr, float* d_germ_val,
                                  uint8_t* d_germ_state, uint32_t* d_count, uint32_t* d_nrec, cudaStream_t st) {
    cudaError_t e = as_launch_twin_heads(cfg, p0, p1, d_twin_next, d_twin_head, d_heads_scratch, d_counters, st);
    if (e != cudaSuccess) return e;
    return as_launch_noise_twin_groups(d_counts, S, P, p0, p1, d_twin_next, d_heads_scratch, d_counters, C, cut, d_thr, d_germ_val,
                                       d_germ_state, d_count, d_nrec, st);
}

cudaError_t as_launch_widen16(const uint16_t* d_in, uint32_t* d_out, int64_t n_words, cudaStream_t st) {
    if (n_words <= 0) return cudaSuccess;
    widen16_kernel<<<cdiv64(n_words, 256), 256, 0, st>>>(reinterpret_cast<const uint2*>(d_in), reinterpret_cast<uint4*>(d_out),
                                                        n_words);
    return cudaGetLastError();
}

cudaError_t as_launch_unpack(const uint32_t* d_in, uint32_t* d_out, int64_t n_words, cudaStream_t st) {
    if (n_words <= 0) return cudaSuccess;
    unpack_kernel<<<cdiv64(n_words, 256), 256, 0, st>>>(d_in, reinterpret_cast<uint4*>(d_out), n_words);
    return cudaGetLastError();
}

cudaError_t as_launch_patch_wide(const as_wide_record* d_wide, int64_t m, uint32_t* d_tile, int64_t n, int64_t p0,
                                 int n_samples, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    patch_wide_kernel<<<cdiv64(m, 128), 128, 0, st>>>(d_wide, m, reinterpret_cast<uint4*>(d_tile), n, p0, n_samples);
    return cudaGetLastError();
}

cudaError_t as_launch_thr_view(const float* d_thr, float* d_view, int64_t n, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    thr_view_kernel<<<cdiv64((n + 3) / 4, 256), 256, 0, st>>>(d_thr, d_view, n);
    return cudaGetLastError();
}

int as_call_chunk(int T, int64_t n_slots) {
    // tumour samples per CTA.  Enough CTAs for about ten waves of the 148 x 5 resident ones (a short tail even when
    // CTAs run for milliseconds), but at least 16 samples = 4 stages per CTA (its pipeline fill is a fixed cost).
    // Measured: 41 k slots x 96 tumours 64 -> 50 us; 100 k x 10,000 unchanged; 2 M x 500 is one chunk either way.
    const int64_t tiles = (n_slots + AS_TILE_SLOTS - 1) / AS_TILE_SLOTS;
    const int64_t chunks = std::max<int64_t>(1, (148ll * 5 * 10 + tiles - 1) / std::max<int64_t>(tiles, 1));
    int64_t chunk = (T + chunks - 1) / chunks;
    if (chunk < 16) chunk = 16;
    if (chunk > T) chunk = T;
    while ((T + chunk - 1) / chunk > 65535) chunk *= 2;  // gridDim.y limit
    return (int)(chunk < 1 ? 1 : chunk);
}

template <int K, int STAGES, bool PRE, bool SWEEP>
static cudaError_t launch_call_staged_impl(dim3 grid, const uint4* c, int T, int64_t P, int64_t p0, int64_t p1, int chunk,
                                      const uint8_t* ref, const float* tv, int n_c, int64_t c_stride, uint32_t cut,
                                      as_call* calls, int64_t cap, unsigned long long* n, cudaStream_t st) {
    static bool configured[AS_MAX_DEVICES] = {};  // the attribute is per device
    const int smem = StageRing<K, STAGES>::kStageBytes * STAGES;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= AS_MAX_DEVICES || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(call_staged_kernel<K, STAGES, PRE, SWEEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < AS_MAX_DEVICES) configured[dev] = true;
    }
    call_staged_kernel<K, STAGES, PRE, SWEEP><<<grid, AS_CTA_THREADS, smem, st>>>(c, T, P, p0, p1, chunk, ref, tv, n_c, c_stride, cut, calls,
                                                                           cap, n);
    return cudaGetLastError();
}

template <int K, int STAGES, int D>
static cudaError_t launch_call_forward(dim3 grid, const uint4* c, int T, int64_t P, int64_t p0, int64_t p1, int chunk,
                                       const uint8_t* ref, const float* tv, uint32_t cut, int pend_cap, as_call* calls, int64_t cap,
                                       unsigned long long* n, cudaStream_t st) {
    static bool configured[AS_MAX_DEVICES] = {};  // the attribute is per device
    const int smem = StageRing<K, STAGES, 1>::kStageBytes * STAGES;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= AS_MAX_DEVICES || !configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(call_forward_kernel<K, STAGES, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < AS_MAX_DEVICES) configured[dev] = true;
    }
    call_forward_kernel<K, STAGES, D><<<grid, AS_TILE_SLOTS + 32 * STAGES, smem, st>>>(c, T, P, p0, p1, chunk, ref, tv, cut, pend_cap, calls, cap, n);
    return cudaGetLastError();
}

template <int K, int STAGES, bool PRE = false>
static cudaError_t launch_call_staged(dim3 grid, const uint4* c, int T, int64_t P, int64_t p0, int64_t p1, int chunk,
                                      const uint8_t* ref, const float* tv, int n_c, int64_t c_stride, uint32_t cut,
                                      as_call* calls, int64_t cap, unsigned long long* n, cudaStream_t st) {
    if (n_c == 1) return launch_call_staged_impl<K, STAGES, PRE, false>(grid, c, T, P, p0, p1, chunk, ref, tv, 1, 0, cut, calls, cap, n, st);
    // sweeps run on the default geometry with the pre-screen, whatever variant is selected
    return launch_call_staged_impl<3, 2, true, true>(grid, c, T, P, p0, p1, chunk, ref, tv, n_c, c_stride, cut, calls, cap, n, st);
}

cudaError_t as_launch_call_sweep(int variant, const uint32_t* d_counts, int T, int64_t P, int64_t p0, int64_t p1,
                                 const uint8_t* d_ref, const float* d_thr_views, int n_c, int64_t c_stride, uint32_t cut,
                                 as_call* d_calls, int64_t cap, unsigned long long* d_n_calls, int fwd_pending_cap, cudaStream_t st) {
    if (p1 <= p0 || T <= 0 || n_c <= 0) return cudaSuccess;
    const uint4* c = reinterpret_cast<const uint4*>(d_counts);
    const int chunk = as_call_chunk(T, p1 - p0);
    dim3 grid(cdiv64(p1 - p0, AS_CALL_THREADS), (unsigned)((T + chunk - 1) / chunk));
#define AS_CALL_ARGS c, T, P, p0, p1, chunk, d_ref, d_thr_views, cut, d_calls, cap, d_n_calls
#define AS_SWEEP_ARGS c, T, P, p0, p1, chunk, d_ref, d_thr_views, n_c, c_stride, cut, d_calls, cap, d_n_calls
#define AS_FWD_ARGS c, T, P, p0, p1, chunk, d_ref, d_thr_views, cut, fwd_pending_cap, d_calls, cap, d_n_calls
    switch (variant) {
        case 0: if (n_c != 1) return cudaErrorInvalidValue; call_naive_kernel<<<grid, AS_CALL_THREADS, 0, st>>>(AS_CALL_ARGS); return cudaGetLastError();
        case 1: if (n_c != 1) return cudaErrorInvalidValue; call_queued_kernel<<<grid, AS_CALL_THREADS, 0, st>>>(AS_CALL_ARGS); return cudaGetLastError();
        case 3: return launch_call_staged<4, 2>(grid, AS_SWEEP_ARGS, st);
        case 11: return launch_call_staged<3, 2>(grid, AS_SWEEP_ARGS, st);
        case 14: return launch_call_staged<4, 2, true>(grid, AS_SWEEP_ARGS, st);
        case 15: return launch_call_staged<3, 2, true>(grid, AS_SWEEP_ARGS, st);
        default: if (n_c != 1) break; return launch_call_forward<4, 3, 2>(grid, AS_FWD_ARGS, st);
    }
    // a sweep of several tables on a staged variant: the in-stage sweep kernel
    return launch_call_staged<3, 2, true>(grid, AS_SWEEP_ARGS, st);
#undef AS_CALL_ARGS
#undef AS_SWEEP_ARGS
#undef AS_FWD_ARGS
}

cudaError_t as_launch_call(int variant, const uint32_t* d_counts, int T, int64_t P, int64_t p0, int64_t p1,
                           const uint8_t* d_ref, const float* d_thr_view, uint32_t cut, as_call* d_calls, int64_t cap,
                           unsigned long long* d_n_calls, int fwd_pending_cap, cudaStream_t st) {
    return as_launch_call_sweep(variant, d_counts, T, P, p0, p1, d_ref, d_thr_view, 1, 0, cut, d_calls, cap, d_n_calls, fwd_pending_cap, st);
}

cudaError_t as_launch_poisson_test(const int32_t* k, const int32_t* rd, const float* err, int64_t n, double* p,
                                   double* q, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    poisson_test_kernel<<<cdiv64(n, 128), 128, 0, st>>>(k, rd, err, n, p, q);
    return cudaGetLastError();
}

cudaError_t as_launch_gammaq(const double* s, const double* z, int64_t n, double* out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    gammaq_kernel<<<cdiv64(n, 128), 128, 0, st>>>(s, z, n, out);
    return cudaGetLastError();
}

cudaError_t as_launch_synth_twin_links(int64_t P, const as_synth_params* prm, int32_t* d_twin_next, int32_t* d_twin_head,
                                       cudaStream_t st) {
    if (P <= 0) return cudaSuccess;
    synth_twin_links_kernel<<<cdiv64(P, 256), 256, 0, st>>>(P, *prm, d_twin_next, d_twin_head);
    return cudaGetLastError();
}

cudaError_t as_launch_synth(uint32_t* d_counts, int n_samples, int64_t P, uint8_t* d_ref, const as_synth_params* prm,
                            cudaStream_t st) {
    if (P <= 0 || n_samples <= 0) return cudaSuccess;
    const int64_t target = 148ll * 2048 * 2;
    int64_t ychunks = (target + P - 1) / P;
    if (ychunks < 1) ychunks = 1;
    if (ychunks > n_samples) ychunks = n_samples;
    if (ychunks > 65535) ychunks = 65535;
    dim3 grid(cdiv64(P, 128), (unsigned)ychunks);
    synth_kernel<<<grid, 128, 0, st>>>(reinterpret_cast<uint4*>(d_counts), n_samples, P, d_ref, *prm);
    return cudaGetLastError();
}
