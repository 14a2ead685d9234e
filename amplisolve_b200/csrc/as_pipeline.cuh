// Shared-memory staging of position tiles with the Blackwell bulk-copy engine (TMA, 1-D form).
//
// A CTA owns a tile of AS_TILE_SLOTS consecutive panel slots and walks the sample axis.  One elected
// producer thread streams [K samples][2 strands][tile] blocks (or the forward strand only) of the count tensor into a ring
// of shared-memory stages with cp.async.bulk (SASS: UBLKCP), one 2 KiB copy per (sample, strand) row, each
// stage guarded by a "full" mbarrier (transaction-count completion) and an "empty" mbarrier (one arrival
// per consumer warp).  The consumer warps never touch global memory for counts and hold no in-flight load
// registers, so the memory system sees up to (stages-1) * K * 4 KiB outstanding per CTA regardless of how
// long the arithmetic on a stage takes.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace asdev {

#define AS_TILE_SLOTS 128      /* slots per CTA tile = consumer threads per CTA */
#define AS_CONSUMER_WARPS 4
#define AS_CTA_THREADS (AS_TILE_SLOTS + 32) /* + one producer warp */

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Blocking wait: try_wait parks the warp until the phase completes or the suspend-time hint (ns) runs out, so a waiting
// warp issues one instruction per AS_MBAR_SUSPEND_NS instead of spinning (ncu of round 1: the producer's and the
// consumers' polling loops were 58 % of the warp instructions the sweep caller executed).
#define AS_MBAR_SUSPEND_NS 20000
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity), "r"(AS_MBAR_SUSPEND_NS)
        : "memory");
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier.  bytes % 16 == 0, both 16-B aligned.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// 16-byte asynchronous copy global -> shared through L2 only (SASS: LDGSTS), tracked per thread in commit groups: a thread
// may read what it copied after cp.async.wait_group, other lanes of its warp after a __syncwarp that follows.
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src_gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// wait until at most N of this thread's most recent commit groups are still in flight
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Ring geometry.  A stage holds K samples x STRANDS strands x AS_TILE_SLOTS uint4 words; STRANDS = 1 streams the
// forward strand only (call_forward_kernel, which fetches reverse-strand words on its own and refills stages from its
// control warp with fill() rather than running produce()).
template <int K, int STAGES, int STRANDS = 2>
struct StageRing {
    static_assert(STRANDS == 1 || STRANDS == 2, "one or both strands per sample");
    static constexpr int kStageWords = K * STRANDS * AS_TILE_SLOTS;  // uint4 words
    static constexpr int kStageBytes = kStageWords * 16;
    uint4* data;        // [STAGES][K][STRANDS][AS_TILE_SLOTS]
    uint64_t* full;     // [STAGES]
    uint64_t* empty;    // [STAGES]

    __device__ __forceinline__ void init(void* smem_base, uint64_t* bars) {
        data = reinterpret_cast<uint4*>(smem_base);
        full = bars;
        empty = bars + STAGES;
        if (threadIdx.x == 0) {
            for (int s = 0; s < STAGES; ++s) {
                mbar_init(&full[s], 1);
                mbar_init(&empty[s], AS_CONSUMER_WARPS);
            }
            mbar_init_fence();
        }
        __syncthreads();
    }
    __device__ __forceinline__ const uint4* stage(int s) const { return data + (size_t)s * kStageWords; }

    // One thread: bulk-copy iteration `it` (samples t0 + it*K on, at most up to t1) of the tile whose first word is `src`
    // (= counts + p0) into its stage, which must be free; sample stride `sstride` words, strand stride `P` words,
    // row_bytes = 16 x the valid slots of the tile.
    __device__ __forceinline__ void fill(int it, const uint4* __restrict__ src, int64_t sstride, int64_t P, int t0, int t1,
                                         uint32_t row_bytes) {
        const int s = it % STAGES, t = t0 + it * K;
        const int k = min(K, t1 - t);
        mbar_expect_tx(&full[s], row_bytes * (uint32_t)STRANDS * (uint32_t)k);
        uint4* dst = data + (size_t)s * kStageWords;
        for (int j = 0; j < k; ++j) {
            const uint4* g = src + (int64_t)(t + j) * sstride;
            bulk_g2s(dst + (j * STRANDS + 0) * AS_TILE_SLOTS, g, row_bytes, &full[s]);
            if (STRANDS == 2) bulk_g2s(dst + (j * STRANDS + 1) * AS_TILE_SLOTS, g + P, row_bytes, &full[s]);
        }
    }
    // Producer: one thread.  Streams samples [t0, t1) of the tile, n_slots valid slots in the tile.
    __device__ __forceinline__ void produce(const uint4* __restrict__ src, int64_t sstride, int64_t P, int t0, int t1,
                                            int n_slots) {
        const uint32_t row_bytes = (uint32_t)n_slots * 16u;
        for (int it = 0; t0 + it * K < t1; ++it) {
            if (it >= STAGES) mbar_wait(&empty[it % STAGES], ((it / STAGES) - 1) & 1);
            fill(it, src, sstride, P, t0, t1, row_bytes);
        }
    }
    // Consumer side: wait for iteration `it` to land / hand its stage back (one arrival per warp).
    __device__ __forceinline__ const uint4* consumer_wait(int it) const {
        const int s = it % STAGES;
        mbar_wait(&full[s], (it / STAGES) & 1);
        return data + (size_t)s * kStageWords;
    }
    __device__ __forceinline__ void consumer_release(int it) const {
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(&empty[it % STAGES]);
    }
};

}  // namespace asdev
