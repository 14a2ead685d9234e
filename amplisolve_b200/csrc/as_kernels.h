// Internal: kernel launchers shared between as_kernels.cu and as_capi.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "../../include/amplisolve_b200.h"

#define AS_NOISE_THREADS 128
#define AS_NOISE_UNROLL 4
#define AS_CALL_THREADS 128
#define AS_MAX_DEVICES 64
/* 1: a duplicated position whose two slots share a CTA tile is reduced inside the staged noise kernel: each slot's
 * thread scans its own rows, the two states are merged exactly after the sample loop (as_noise.cuh pair_merge).
 * 0: every twin group goes to noise_pair_kernel / noise_twin_kernel. */
#define AS_INTILE_TWINS 1
#define AS_DEFAULT_CALL_KERNEL 13 /* forward-first (call_forward_kernel): forward plane streamed, 4 samples per stage, 3 stages; four scan warps and one control warp per stage, which extracts the forward candidates, fetches their reverse words and refills its stage; 15 = the both-strand staged caller it replaced */
#define AS_DEFAULT_NOISE_KERNEL 1 /* TMA-staged, 4 samples per stage, 3 stages */
#define AS_DEFERRED_CALL_KERNEL 20 /* scan -> resolve -> series (as_call_deferred.cu); what a sweep runs by default */

cudaError_t as_launch_noise_main(int cfg, const uint32_t* d_counts, int S, int64_t P, int64_t p0, int64_t p1,
                                 const int32_t* d_twin_next, const int32_t* d_twin_head, int64_t twin_base, float C,
                                 uint32_t cut, float* d_thr, float* d_germ_val, uint8_t* d_germ_state,
                                 uint32_t* d_count, uint32_t* d_nrec, cudaStream_t st);
cudaError_t as_launch_noise_twins(int cfg, const uint32_t* d_counts, int S, int64_t P, int64_t p0, int64_t p1,
                                  const int32_t* d_twin_next, const int32_t* d_twin_head, int32_t* d_heads_scratch,
                                  uint32_t* d_nheads_scratch, float C, uint32_t cut, float* d_thr, float* d_germ_val,
                                  uint8_t* d_germ_state, uint32_t* d_count, uint32_t* d_nrec, cudaStream_t st);
cudaError_t as_launch_twin_heads(int cfg, int64_t p0, int64_t p1, const int32_t* d_twin_next, const int32_t* d_twin_head,
                                 int32_t* d_heads_scratch, uint32_t* d_counters, cudaStream_t st);
cudaError_t as_launch_noise_twin_groups(const uint32_t* d_counts, int S, int64_t P, int64_t p0, int64_t p1,
                                        const int32_t* d_twin_next, const int32_t* d_heads_scratch, const uint32_t* d_counters,
                                        float C, uint32_t cut, float* d_thr, float* d_germ_val, uint8_t* d_germ_state,
                                        uint32_t* d_count, uint32_t* d_nrec, cudaStream_t st);
// as_noise_pattern.cu: every output of the noise model for n_c (1..8) values of C in ONE pass over the normals; table c at
// d_thr + c * thr_stride floats.  The ring is (4 samples, 3 stages); geom 0 unrolls the 4 records of a stage, geom 1
// (n_c = 1 and n_c 4..5 only; others run geom 0) walks them one by one.
cudaError_t as_launch_noise_pattern(int geom, const uint32_t* d_counts, int S, int64_t P, int64_t p0, int64_t p1,
                                    const int32_t* d_twin_next, const int32_t* d_twin_head, int64_t twin_base,
                                    const float* c_values, int n_c, uint32_t cut, float* d_thr, int64_t thr_stride,
                                    float* d_germ_val, uint8_t* d_germ_state, uint32_t* d_count, uint32_t* d_nrec, cudaStream_t st);
// as_call_deferred.cu: the caller as scan -> resolve -> series kernels over candidate / survivor lists in d_scratch
size_t as_deferred_scratch_bytes(int T, int64_t n_slots, int64_t cap_override, int64_t* cap_cand, int64_t* cap_surv);
#define AS_DEFER_MAX_CHUNKS 8
int as_deferred_chunks(int64_t n_slots, int want);
cudaError_t as_launch_call_deferred(const uint32_t* d_counts, int T, int64_t P, int64_t p0, int64_t p1, const uint8_t* d_ref,
                                    const float* d_thr_views, int n_c, int64_t c_stride, uint32_t cut, as_call* d_calls,
                                    int64_t cap, unsigned long long* d_n_calls, void* d_scratch, int64_t cap_cand,
                                    int64_t cap_surv, cudaStream_t st, cudaStream_t aux, cudaEvent_t* ev, int n_chunks);
cudaError_t as_launch_widen16(const uint16_t* d_in, uint32_t* d_out, int64_t n_words, cudaStream_t st);
cudaError_t as_launch_unpack(const uint32_t* d_in, uint32_t* d_out, int64_t n_words, cudaStream_t st);
cudaError_t as_launch_patch_wide(const as_wide_record* d_wide, int64_t m, uint32_t* d_tile, int64_t n, int64_t p0,
                                 int n_samples, cudaStream_t st);
cudaError_t as_launch_thr_view(const float* d_thr, float* d_view, int64_t n, cudaStream_t st);
int as_call_chunk(int T, int64_t n_slots);
// fwd_pending_cap: usable depth of call_forward_kernel's per-CTA pending ring, 1..AS_FWD_PENDING (else the whole ring)
#define AS_FWD_PENDING 128
cudaError_t as_launch_call(int variant, const uint32_t* d_counts, int T, int64_t P, int64_t p0, int64_t p1,
                           const uint8_t* d_ref, const float* d_thr_view, uint32_t cut, as_call* d_calls, int64_t cap,
                           unsigned long long* d_n_calls, int fwd_pending_cap, cudaStream_t st);
// as_sort.cu: call list housekeeping of the _host caller pipeline
cudaError_t as_launch_call_slot_offset(as_call* d_calls, const unsigned long long* d_n_prev, const unsigned long long* d_n_now,
                                       int64_t cap, int32_t off, cudaStream_t st);
size_t as_sort_calls_scratch_bytes(int64_t n);
cudaError_t as_launch_sort_calls(const as_call* d_calls, int64_t n, as_call* d_sorted, void* d_scratch, size_t scratch_bytes,
                                 cudaStream_t st);
// as_fisher.cu: Fisher strand-bias tests, one warp per table {FW, BW, alt_fw, alt_bw}; d_lg[i] = lgamma(i + 1)
cudaError_t as_launch_fisher(const int32_t* d_tables, int64_t n, const double* d_lg, double* d_p, cudaStream_t st);
// n_c threshold tables c_stride floats apart (noise-floor sweep): list ci at d_calls + ci * cap, counter d_n_calls[ci]
cudaError_t as_launch_call_sweep(int variant, const uint32_t* d_counts, int T, int64_t P, int64_t p0, int64_t p1,
                                 const uint8_t* d_ref, const float* d_thr_views, int n_c, int64_t c_stride, uint32_t cut,
                                 as_call* d_calls, int64_t cap, unsigned long long* d_n_calls, int fwd_pending_cap, cudaStream_t st);
// as_pileup.cu: BAM records -> counts[2][P][4] of one sample (SURVEY.md 8 f4); stats[0] reads used, stats[1] bases counted
cudaError_t as_launch_pileup(const uint8_t* d_rec, const int64_t* d_rec_off, int64_t n_rec, int64_t n_bytes,
                             const int32_t* d_ref_contig, int32_t n_ref, const int64_t* d_contig_first,
                             const int32_t* d_slot_pos, int64_t P, int32_t mbq, int32_t mrq, uint32_t skip_flags,
                             uint32_t* d_counts, unsigned long long* d_stats, cudaStream_t st);
// counts [2][U][4] of one sample -> its wire slice: fmt 1 packed [2][P] uint32, fmt 2 uint16 [2][P][4]; slot s takes
// position d_slot_unique[s], a depth below mdc is absent; escaped records -> d_wide (at most cap kept), d_n[0] = escaped,
// d_n[1] += present slots (zero d_n first)
cudaError_t as_launch_pileup_encode(int fmt, const uint32_t* d_counts, int64_t U, const int32_t* d_slot_unique, int64_t P,
                                    int32_t mdc, int32_t sample, void* d_wire, as_wide_record* d_wide, int64_t cap,
                                    unsigned long long* d_n, cudaStream_t st);
// as_sites.cu: site_test_kernel over counts [T][2][H][4]; site_ra[h] = ref | alt << 8, thr [n_c][H][2], out [n_c][T][H]
cudaError_t as_launch_site_test(const uint32_t* d_counts, int T, int H, const uint16_t* d_site_ra, const float* d_thr, int n_c,
                                uint32_t cut, as_site_test* d_out, cudaStream_t st);
cudaError_t as_launch_poisson_test(const int32_t* k, const int32_t* rd, const float* err, int64_t n, double* p,
                                   double* q, cudaStream_t st);
cudaError_t as_launch_gammaq(const double* s, const double* z, int64_t n, double* out, cudaStream_t st);
cudaError_t as_launch_synth_twin_links(int64_t P, const as_synth_params* prm, int32_t* d_twin_next, int32_t* d_twin_head,
                                       cudaStream_t st);
cudaError_t as_launch_synth(uint32_t* d_counts, int n_samples, int64_t P, uint8_t* d_ref, const as_synth_params* prm,
                            cudaStream_t st);
