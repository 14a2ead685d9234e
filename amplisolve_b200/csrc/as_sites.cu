// Site report: the Poisson strand tests of listed (slot, alt) sites in every tumour, called or not (as_site_tests_host*).
//   VC = source_codes/AmpliSolveVariantCalling.cpp of the reference.
// The reference computes Q_fw and Q_bw for every row and alt (VC:895-896) and only then applies the decision of VC:898; the
// caller kernels skip every evaluation that cannot end in a call.  This kernel evaluates all of them, through the same
// device functions (poisson_p, q_at_least_5 of as_device.cuh), so that its CALLED status is the caller's decision bit for bit.
#include "as_device.cuh"
#include "as_kernels.h"

using namespace asdev;

#define AS_SITE_THREADS 256

// One lane per (table, site, sample, strand); the two strands of an entry are neighbouring lanes and trade depth, presence
// and p by shuffle.  Samples run fastest, so a warp holds 16 samples of ONE site and table: the same threshold and similar
// depths, hence the same incomplete-gamma branch and similar iteration counts in all its lanes.  A lane with k = 0 returns
// p = 1 at once (VC:3858-3861).
//   counts [T][2][H][4]: the records of the H sites' slots; site_ra[h] = ref | alt << 8; thr [n_c][H][2] = the caller views
//   (forward, reverse) of (site slot, alt) in table c; out [n_c][T][H].
__global__ void __launch_bounds__(AS_SITE_THREADS)
site_test_kernel(const uint4* __restrict__ counts, int T, int H, const uint16_t* __restrict__ site_ra, const float2* __restrict__ thr,
                 int n_c, uint32_t cut, as_site_test* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * AS_SITE_THREADS + threadIdx.x;
    const int64_t total = (int64_t)n_c * H * T * 2;
    const bool live = i < total;  // total is even: both lanes of an entry are live or neither is
    const int strand = (int)(i & 1);
    const int64_t e = i >> 1;
    const int t = live ? (int)(e % T) : 0;
    const int64_t ch = live ? e / T : 0;
    const int h = (int)(ch % H), c = (int)(ch / H);
    uint32_t depth = 0, k = 0, absent = 1, ref = 4, alt = 0;
    float err = 0.0f;
    if (live) {
        const uint4 r = counts[((int64_t)t * 2 + strand) * H + h];
        const uint16_t ra = site_ra[h];
        ref = ra & 0xFFu;
        alt = ra >> 8;
        const float2 tv = thr[(int64_t)c * H + h];
        err = strand == 0 ? tv.x : tv.y;
        absent = (int32_t)r.x < 0 ? 1u : 0u;  // the caller's test of the forward word (VC:723: no ASEQ row)
        if (!absent) {
            depth = r.x + r.y + r.z + r.w;  // VC:760-770
            k = comp(r, (int)alt);
        }
    }
    absent = __shfl_sync(0xffffffffu, absent, threadIdx.x & ~1);  // the forward lane's word decides, as in the caller
    const uint32_t depth_other = __shfl_xor_sync(0xffffffffu, depth, 1), k_other = __shfl_xor_sync(0xffffffffu, k, 1);
    const bool testable = ref <= 3u && alt != ref;  // VC:3290-3293; the reference tests the three other bases only
    double p = __longlong_as_double(0x7FF8000000000000ll);  // NaN: not evaluated
    if (live && !absent && testable && err != -1.0f)  // err -1: the reference's Q is -888 (VC:3844-3849), never a call
        p = poisson_p((int)k, (int)depth, err);         // VC:895 / VC:896, no screen
    const double p_other = __shfl_xor_sync(0xffffffffu, p, 1);
    if (!live || strand != 0) return;
    as_site_test o;
    o.depth_fw = depth; o.depth_bw = depth_other;
    o.alt_fw = k; o.alt_bw = k_other;
    o.p_fw = p; o.p_bw = p_other;
    o.pad = 0;
    if (absent) { o.status = AS_SITE_NO_DATA; o.depth_fw = o.depth_bw = o.alt_fw = o.alt_bw = 0; }
    else if (!testable) o.status = AS_SITE_NOT_TESTABLE;
    else if (!(depth >= cut && depth_other >= cut)) o.status = AS_SITE_LOW_COVERAGE;  // VC:898
    else o.status = (q_at_least_5(p) && q_at_least_5(p_other)) ? AS_SITE_CALLED : AS_SITE_NOT_CALLED;  // VC:898
    out[((int64_t)c * T + t) * H + h] = o;
}

cudaError_t as_launch_site_test(const uint32_t* d_counts, int T, int H, const uint16_t* d_site_ra, const float* d_thr, int n_c,
                                uint32_t cut, as_site_test* d_out, cudaStream_t st) {
    const int64_t lanes = (int64_t)n_c * H * T * 2;
    if (lanes <= 0) return cudaSuccess;
    const int64_t blocks = (lanes + AS_SITE_THREADS - 1) / AS_SITE_THREADS;
    if (blocks > 0x7FFFFFFFll) return cudaErrorInvalidValue;
    site_test_kernel<<<(unsigned)blocks, AS_SITE_THREADS, 0, st>>>(reinterpret_cast<const uint4*>(d_counts), T, H, d_site_ra,
                                                                  reinterpret_cast<const float2*>(d_thr), n_c, cut, d_out);
    return cudaGetLastError();
}
