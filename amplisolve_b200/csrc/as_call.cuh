// Device helpers shared by the caller kernels (as_kernels.cu: in-stage and forward-first callers; as_call_deferred.cu:
// scan / resolve / series pipeline): the two exact screens, the integer pre-screen of the scan and the survivor entry.
//   VC = source_codes/AmpliSolveVariantCalling.cpp of the reference.
#pragma once
#include "as_device.cuh"

namespace asdev {

// exact screen of SURVEY.md B.6(3): on the continued-fraction branch of VC:3728 (m >= k and m > 1) the
// reference's Q never reaches 5 (p = P(X >= k) >= 1/2 for a Poisson mean m >= k; validated against the
// compiled reference including the region where its 99-step cap leaves the fraction unconverged,
// tests/test_oracle_golden.py::test_screen_continued_fraction_branch_never_calls), so such a strand test can only veto the call.
//
// Second exact screen, for small k: p = P(X >= k | m) grows with m, so there is a critical mean m*(k) with
// p(k, m*) = P* (the largest p whose Q reaches 5, as_device.cuh) and a strand test with m above it cannot pass.
// AS_MCRIT[k-1] = m*(k) * (1 + 1e-9), k = 1..64, m* solved to 40 digits (mpmath; scripts/critical_means.py).  Between
// m*(k) and k the reference evaluates the series of VC:3785-3794 (z < s), whose p is within 1.5e-13 relative of the exact
// value there (measured against mpmath over k = 1..64); the 1e-9 margin in m is a margin of >= 5e-10 relative in p, so
// m >= AS_MCRIT[k-1] implies that the reference's own p exceeds P*.  Pairs inside the margin go to the series as before.
// This matters where depth * e is of order 1 (low noise floors, shallow positions): there "m >= k" never fires and
// every candidate with one or two alt reads would otherwise cost a full fp64 series only to be rejected.
__device__ const double AS_MCRIT[64] = {
    0.3801304084463019, 1.1417568666028408, 1.9737827925528142, 2.836655303617698,
    3.717842035557975, 4.6115129863431354, 5.514398678438836, 6.4244483020565735,
    7.340275226714001, 8.26088993116463, 9.185556927304383, 10.113711843311759,
    11.044910368246212, 11.978795260900911, 12.915074175299806, 13.853504259954532,
    14.793881161100241, 15.736030981805042, 16.679804280096405, 17.62507150754917,
    18.571719486996063, 19.519648653852276, 20.468770867935323, 21.419007657863915,
    22.370288797876483, 23.322551143218725, 24.275737668892344, 25.229796669971126,
    26.184681091478662, 27.14034796305633, 28.096757919060714, 29.05387478882073,
    30.01166524490941, 30.97009849969475, 31.929146042307917, 32.888781409637,
    33.84897998611586, 34.80971882800224, 35.77097650858012, 36.73273298131915,
    37.694969458508524, 38.657668303278726, 39.62081293324896, 40.58438773430595,
    41.548377983241544, 42.51276977816144, 43.4775499757315, 44.44270613445805,
    45.40822646330781, 46.37409977506551, 47.34031544390594, 48.30686336672417,
    49.273733927824765, 50.240917966620174, 51.208406748030676, 52.17619193531465,
    53.14426556508969, 54.11262002433242, 55.08124802916871, 56.05014260528682,
    57.019297069824276, 57.988705014595105, 58.95836029053817, 59.92825699327966,
};

__device__ __forceinline__ bool strand_can_pass(uint32_t k, uint32_t depth, float err) {
    if (err == -1.0f) return false;  // VC:3844-3849: Q = -888
    const double m = __dmul_rn((double)depth, (double)effective_err(err));
    if (m >= (double)k && m > 1.0) return false;
    if (k >= 1u && k <= 64u && m >= AS_MCRIT[k - 1u]) return false;
    return true;
}

// Integer pre-screen of the staged caller's scan.  R = floor(e_min * 2^32) for the smallest threshold e_min of the strand;
// m16 = floor(16 * depth * e_min) in sixteenths (depth saturates at 2^28: a smaller product is still a lower bound).
// Returns K such that a strand test with 1 <= k <= K cannot pass for any alt base (real mean m >= m16 / 16):
//   K = floor(m16/16 + 9/16) when that is <= 64: m >= K - 9/16 >= m*(K)(1 + 1e-9) = AS_MCRIT[K-1] (checked for K = 1..64 in
//       tests/test_host_cpu.py), the critical-mean screen of strand_can_pass;
//   K = floor(m16/16) otherwise: m >= k and m > 1, the continued-fraction screen.
// floor((m16 + 9) / 16) <= 64 exactly when m16 <= 1030, so the two cases are one add under a compare (no overflow: the 9 is
// only added to small values) -- four instructions per bound, which matters where the scan evaluates one per alt base.
__device__ __forceinline__ uint32_t prescreen_k(uint32_t depth, uint32_t R) {
    const uint32_t d16 = depth > 0x0FFFFFFFu ? 0xFFFFFFFFu : depth << 4;
    const uint32_t m16 = __umulhi(d16, R);
    return (m16 + (m16 <= 1030u ? 9u : 0u)) >> 4;
}

// Survivor entry of the staged kernel: 24 bytes (the thresholds are read again from thr_view when the series is
// evaluated -- survivors are a few per ten thousand records -- so that five CTAs fit one SM).
struct StagedCand {
    uint32_t k_fw, d_fw, k_bw, d_bw;
    uint32_t sample_alt;  // sample | threshold table (noise-floor sweep) << 27 | alt << 30
    int32_t slot;
};
static_assert(sizeof(StagedCand) == 24, "StagedCand is three 8-byte words");

}  // namespace asdev
