// BAM records -> strand-specific base counts per panel position (SURVEY.md §8 f4: the computeCounts / ASEQ PILEUP step
// that produces the *.PILEUP.ASEQ files both reference programs start from; Execution_examples.md:16-54).
//
// The reference ships that step as a binary only (Pre-compiled_binaries/computeCounts, Mach-O), so there is no source to
// restate: this is a NEW design with the conventions of a samtools-style pileup, stated here and in DESIGN.md §9, and
// checked against oracle/pileup_oracle.py (parity with the binary: UNPINNED).
//   * a read is used when  mapq >= mrq  and none of its flag bits is in skip_flags
//     (default 0x704: unmapped, secondary, QC fail, duplicate);
//   * a base is counted when its CIGAR op aligns it to the reference (M, =, X), its quality is >= mbq (a record without
//     qualities, 0xFF, counts), and it is A, C, G or T;  deletions, reference skips, insertions, clips count nothing;
//   * strand = flag 0x10;  counts[strand][slot][base] is exactly the layout of the count tensor of one sample
//     (include/amplisolve_b200.h), so a pileup feeds the noise model / caller without a text file in between: the two
//     programs read a directory of BAM files through pileup_encode_kernel (as_pileup_end_wire).
//
// Input: the UNCOMPRESSED record stream of a BAM file (what BGZF inflates to, header stripped) and the byte offset of
// every record; the panel as sorted 0-based positions per contig.  One warp per read: the CIGAR is walked by the whole
// warp (uniform); for an aligned block the range of panel slots under it is found by two binary searches and the lanes
// walk those slots (not the read's bases: a base outside the panel costs nothing).
//
// pileup_encode_kernel (below) turns the counts of one sample into its slice of the programs' host wire tensor.
#include "as_kernels.h"
#include "as_wire.h"

#include <cuda_runtime.h>
#include <stdint.h>

namespace asdev {

__device__ __forceinline__ uint32_t rd_u32(const uint8_t* p) {  // BAM records are not aligned
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__device__ __forceinline__ uint32_t rd_u16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

// first index in [lo, hi) with pos[index] >= key (32-bit indices: pos is the slice of one contig)
__device__ __forceinline__ uint32_t lower_bound_pos(const int32_t* __restrict__ pos, uint32_t lo, uint32_t hi, int32_t key) {
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (pos[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(256)
pileup_kernel(const uint8_t* __restrict__ rec, const int64_t* __restrict__ rec_off, int64_t n_rec, int64_t n_bytes,
              const int32_t* __restrict__ ref_contig, int32_t n_ref, const int64_t* __restrict__ contig_first,
              const int32_t* __restrict__ slot_pos, int64_t P, int32_t mbq, int32_t mrq, uint32_t skip_flags,
              uint32_t* __restrict__ counts, unsigned long long* __restrict__ stats) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    unsigned long long used_reads = 0, used_bases = 0;
    for (int64_t r = warp0; r < n_rec; r += n_warps) {
        const uint8_t* b = rec + rec_off[r];  // points at block_size
        const int64_t room = n_bytes - rec_off[r];
        if (room < 36) continue;
        const uint32_t block_size = rd_u32(b);
        if ((int64_t)block_size + 4 > room || block_size < 32) continue;  // truncated record: ignored (the host reports it)
        const int32_t ref_id = (int32_t)rd_u32(b + 4);
        const int32_t pos = (int32_t)rd_u32(b + 8);
        const uint32_t l_name = b[12], mapq = b[13];
        const uint32_t n_cig = rd_u16(b + 16), flag = rd_u16(b + 18);
        const uint32_t l_seq = rd_u32(b + 20);
        if (ref_id < 0 || ref_id >= n_ref || pos < 0) continue;
        if ((flag & skip_flags) != 0u || (int32_t)mapq < mrq) continue;
        const int32_t contig = ref_contig[ref_id];
        if (contig < 0) continue;
        const uint8_t* cig = b + 36 + l_name;
        const uint8_t* seq = cig + 4 * (size_t)n_cig;
        const uint8_t* qual = seq + ((l_seq + 1) >> 1);
        if ((int64_t)(36 + l_name + 4 * (size_t)n_cig + ((l_seq + 1) >> 1) + l_seq) > (int64_t)block_size + 4) continue;
        const int64_t c0 = contig_first[contig];
        const uint32_t n_c = (uint32_t)(contig_first[contig + 1] - c0);  // slots of this contig
        if (n_c == 0u) continue;
        const int32_t* __restrict__ cpos = slot_pos + c0;
        uint32_t* __restrict__ ccounts = counts + ((flag & 0x10u) ? P : 0) * 4 + c0 * 4;  // this strand, this contig
        uint32_t q = 0;      // query offset
        int32_t g = pos;     // reference offset (0-based)
        bool any = false;
        for (uint32_t k = 0; k < n_cig; ++k) {
            const uint32_t v = rd_u32(cig + 4 * (size_t)k);
            const uint32_t op = v & 15u, len = v >> 4;
            if (op == 0u || op == 7u || op == 8u) {  // M, =, X: aligned bases
                if (q + len > l_seq) break;          // malformed
                if (g <= cpos[n_c - 1] && g + (int32_t)len > cpos[0]) {
                    // the panel positions under this block are cpos[j_lo, j_hi): two searches per block (the second over
                    // at most len entries), then the lanes walk those SLOTS -- no lane is spent on a base outside the panel
                    const uint32_t j_lo = lower_bound_pos(cpos, 0u, n_c, g);
                    const uint32_t j_end = n_c - j_lo > len ? j_lo + len : n_c;
                    const uint32_t j_hi = lower_bound_pos(cpos, j_lo, j_end, g + (int32_t)len);
                    for (uint32_t j = j_lo + lane; j < j_hi; j += 32) {
                        const uint32_t qi = q + (uint32_t)(cpos[j] - g);
                        if ((int32_t)qual[qi] < mbq) continue;
                        const uint32_t code = (seq[qi >> 1] >> ((qi & 1u) ? 0 : 4)) & 15u;  // 1, 2, 4, 8 = A, C, G, T
                        if (code == 0u || (code & (code - 1u)) != 0u) continue;               // =, N and the ambiguity codes
                        atomicAdd(&ccounts[(size_t)j * 4 + (__ffs((int)code) - 1)], 1u);
                        used_bases += 1;
                        any = true;
                    }
                }
                q += len; g += (int32_t)len;
            } else if (op == 1u || op == 4u) {  // I, S: query only
                q += len;
            } else if (op == 2u || op == 3u) {  // D, N: reference only
                g += (int32_t)len;
            }  // H, P: neither
        }
        if (__any_sync(0xFFFFFFFFu, any) && lane == 0) used_reads += 1;
    }
    if (stats != nullptr) {
        for (int d = 16; d > 0; d >>= 1) {
            used_reads += __shfl_down_sync(0xFFFFFFFFu, used_reads, d);
            used_bases += __shfl_down_sync(0xFFFFFFFFu, used_bases, d);
        }
        if (lane == 0 && (used_reads | used_bases)) {
            atomicAdd(&stats[0], used_reads);
            atomicAdd(&stats[1], used_bases);
        }
    }
}

// The pileup of one sample -> that sample's slice of a host wire tensor (include/amplisolve_b200.h), so the two programs
// read BAM files without ASEQ text in between.  counts [2][U][4] over the U unique panel positions; slot s of the panel
// takes the record of position slot_unique[s] (twin slots share one); a slot whose depth (64-bit sum of its eight counts,
// as computeCounts sums it) is below mdc is ABSENT.  FMT 1: packed words [2][P] (as_pack_word); FMT 2: uint16 [2][P][4]
// (escaped when a count is >= AS_WIRE_ESCAPE).  Escaped records go to wide[] by warp-ballot compaction (one atomic per
// warp; n[0] counts all of them, entries beyond cap are dropped), present slots to n[1].  One thread per slot.
template <int FMT>
__global__ void __launch_bounds__(256)
pileup_encode_kernel(const uint32_t* __restrict__ counts, int64_t U, const int32_t* __restrict__ slot_unique, int64_t P,
                     int32_t mdc, int32_t sample, void* __restrict__ wire, as_wide_record* __restrict__ wide, int64_t cap,
                     unsigned long long* __restrict__ n) {
    const int lane = threadIdx.x & 31;
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool present = false, escape = false;
    uint32_t f[4] = {0u, 0u, 0u, 0u}, b[4] = {0u, 0u, 0u, 0u};
    if (s < P) {
        const int64_t u = slot_unique[s];
        const uint4 fv = reinterpret_cast<const uint4*>(counts)[u];
        const uint4 bv = reinterpret_cast<const uint4*>(counts)[U + u];
        f[0] = fv.x; f[1] = fv.y; f[2] = fv.z; f[3] = fv.w;
        b[0] = bv.x; b[1] = bv.y; b[2] = bv.z; b[3] = bv.w;
        const unsigned long long depth = (unsigned long long)f[0] + f[1] + f[2] + f[3] + b[0] + b[1] + b[2] + b[3];
        present = depth >= (unsigned long long)(mdc > 0 ? mdc : 0);
        if (FMT == 1) {
            uint32_t* w = static_cast<uint32_t*>(wire);
            uint32_t wf = AS_PACKED_ABSENT, wb = AS_PACKED_ABSENT;
            if (present) {
                escape = !(as_pack_word(f, &wf) && as_pack_word(b, &wb));
                if (escape) wf = wb = AS_PACKED_ESCAPE;
            }
            w[s] = wf;
            w[P + s] = wb;
        } else {
            uint2* w = static_cast<uint2*>(wire);  // four uint16 counts = 8 bytes per (strand, slot)
            uint2 wf = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu), wb = wf;  // AS_WIRE_ABSENT in all four
            if (present) {
                escape = !(as_wire16_fits(f) && as_wire16_fits(b));
                if (escape) {
                    wf = wb = make_uint2(0xFFFEFFFEu, 0xFFFEFFFEu);  // AS_WIRE_ESCAPE in all four
                } else {
                    wf = make_uint2(f[0] | f[1] << 16, f[2] | f[3] << 16);
                    wb = make_uint2(b[0] | b[1] << 16, b[2] | b[3] << 16);
                }
            }
            w[s] = wf;
            w[P + s] = wb;
        }
    }
    const unsigned esc = __ballot_sync(0xFFFFFFFFu, escape);
    const unsigned pre = __ballot_sync(0xFFFFFFFFu, present);
    unsigned long long base = 0;
    if (lane == 0) {
        if (esc) base = atomicAdd(&n[0], (unsigned long long)__popc(esc));
        if (pre) atomicAdd(&n[1], (unsigned long long)__popc(pre));
    }
    base = __shfl_sync(0xFFFFFFFFu, base, 0);
    if (escape) {
        const unsigned long long k = base + (unsigned long long)__popc(esc & ((1u << lane) - 1u));
        if ((int64_t)k < cap) {
            as_wide_record r;
            r.sample = sample;
            r.slot = (int32_t)s;
            for (int i = 0; i < 4; ++i) { r.fw[i] = f[i]; r.bw[i] = b[i]; }
            wide[k] = r;
        }
    }
}

}  // namespace asdev

using namespace asdev;

cudaError_t as_launch_pileup_encode(int fmt, const uint32_t* d_counts, int64_t U, const int32_t* d_slot_unique, int64_t P,
                                    int32_t mdc, int32_t sample, void* d_wire, as_wide_record* d_wide, int64_t cap,
                                    unsigned long long* d_n, cudaStream_t st) {
    if (P <= 0) return cudaSuccess;
    const int threads = 256;
    const unsigned blocks = (unsigned)((P + threads - 1) / threads);
    if (fmt == 1)
        pileup_encode_kernel<1><<<blocks, threads, 0, st>>>(d_counts, U, d_slot_unique, P, mdc, sample, d_wire, d_wide, cap, d_n);
    else
        pileup_encode_kernel<2><<<blocks, threads, 0, st>>>(d_counts, U, d_slot_unique, P, mdc, sample, d_wire, d_wide, cap, d_n);
    return cudaGetLastError();
}

cudaError_t as_launch_pileup(const uint8_t* d_rec, const int64_t* d_rec_off, int64_t n_rec, int64_t n_bytes,
                             const int32_t* d_ref_contig, int32_t n_ref, const int64_t* d_contig_first,
                             const int32_t* d_slot_pos, int64_t P, int32_t mbq, int32_t mrq, uint32_t skip_flags,
                             uint32_t* d_counts, unsigned long long* d_stats, cudaStream_t st) {
    if (n_rec <= 0 || P <= 0) return cudaSuccess;
    const int threads = 256;
    const int64_t want = (n_rec * 32 + threads - 1) / threads;
    const int blocks = (int)(want < 148 * 8 ? want : 148 * 8);  // 8 CTAs of 8 warps per SM, reads strided over the warps
    pileup_kernel<<<blocks, threads, 0, st>>>(d_rec, d_rec_off, n_rec, n_bytes, d_ref_contig, n_ref, d_contig_first, d_slot_pos, P,
                                              mbq, mrq, skip_flags, d_counts, d_stats);
    return cudaGetLastError();
}
