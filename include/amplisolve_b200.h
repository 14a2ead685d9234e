/* amplisolve_b200 -- C ABI of the B200-native AmpliSolve hot path (libamplisolve_b200.so).
 *
 * The reference (dkleftogi/AmpliSolve) has no library or FFI surface: its boundary is the process
 * boundary of two single-file programs.  This header is the boundary a maintainer would bind
 * instead; every entry point names the reference code it replaces
 *   EE = source_codes/AmpliSolveErrorEstimation.cpp, VC = source_codes/AmpliSolveVariantCalling.cpp.
 * The two drop-in executables (amplisolve_b200/bin/AmpliSolveErrorEstimation, ...VariantCalling)
 * and the Python mirror (amplisolve_b200/api.py) are thin callers of exactly these functions.
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success or a negative AS_E* code, with a
 *     human-readable message available from as_last_error() (thread-local).
 *   - there is NO CPU fallback: every compute entry point fails with AS_ECUDA when no sm_100
 *     device / driver is available.
 *   - "_host" entry points take host pointers (pinned or pageable) and do H2D, kernels and D2H
 *     themselves, tiling over slots with double-buffered streams; "_dev" entry points take
 *     device pointers (inputs resident in HBM) and only enqueue kernels on `stream`
 *     (a cudaStream_t passed as void*; NULL = the legacy default stream).  They use scratch owned by the
 *     context (twin-group lists, candidate lists of a sweep): enqueue the _dev calls of ONE context on ONE
 *     stream, or synchronise between calls that go to different streams; use one context per thread.
 *
 * Data layout ("count tensor"): uint32 counts[sample][strand][slot][base]
 *     strand 0 = forward, 1 = reverse; base 0..3 = A,C,G,T; one 16-byte word per (sample,strand,slot),
 *     so the tensor base must be 16-byte aligned.
 *     slot   = index into the BED enumeration of the panel (both ends inclusive, duplicated
 *              positions kept as separate slots: EE:637, EE:2606).
 *     A (sample,slot) with no ASEQ row is ABSENT: all eight words = AS_ABSENT (0xFFFFFFFF).  This is
 *     not the same as a row of zeros: absence changes N in the 0.338*N rule (EE:1742).  Valid counts
 *     are < 2^31 (the reference reads them with %d).
 *     Derivation from an ASEQ row (EE:1149-1176, VC:752-770): fw[b] = X - X_rs, bw[b] = X_rs; the RD
 *     column equals the sum of the eight words in every row the reference's own pileup step writes (the
 *     programs still accept a row where it does not: the error estimation warns, the caller uses the
 *     column as the reference does).  A BAM file
 *     yields the same record without text in between (as_pileup_end_wire below).
 *   Twin slots: a position enumerated by two overlapping amplicons owns several slots.  The
 *     reference keys records by "chrom_pos" text, so all rows of all twins feed one noise estimate
 *     (EE:1241-1245).  twin_next[slot] = next slot of the same position (or -1); twin_head[slot] =
 *     first slot of the position (== slot for singletons).  Both may be NULL (no duplicated position).
 */
#ifndef AMPLISOLVE_B200_H
#define AMPLISOLVE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AS_ABSENT 0xFFFFFFFFu

enum {
    AS_OK = 0,
    AS_EINVAL = -1,   /* bad argument */
    AS_ECUDA = -2,    /* CUDA error, or no usable sm_100 device */
    AS_ENOMEM = -3,
    AS_EIO = -4,      /* file could not be opened / parsed */
    AS_EOVERFLOW = -5 /* call list capacity exceeded (n_calls still reports the true count) */
};

typedef struct as_ctx as_ctx; /* one context per device (as_create) or per device list (as_create_multi); not thread-safe, use one per thread */

/* A called variant as the device emits it.  Replaces the decision of VC:898 plus the two strand
 * tests of VC:895-896.  48 bytes. */
typedef struct {
    int32_t sample; /* index into the tumour axis of the count tensor */
    int32_t slot;   /* panel slot */
    int32_t alt;    /* 0..3 = A,C,G,T */
    int32_t ref;    /* 0..3 */
    double p_fw;    /* the double p-value of VC:3858-3866, forward strand */
    double p_bw;    /* reverse strand */
    double q_fw;    /* Qscore_fw of VC:3868-3882 evaluated in fp64 (100 when p < 1e-10) */
    double q_bw;
} as_call;

/* ---- context ------------------------------------------------------------------------------ */
const char* as_last_error(void);
const char* as_version(void);
int as_device_count(int* n);
int as_create(int device, as_ctx** out);
/* One context over ndev GPUs of the box (BASELINE north_star: "positions shard naturally across the 8 GPUs of one box, with no
 * NCCL on the math path and only a final gather of compacted calls").  The _host entry points split the panel's slots
 * into ndev contiguous ranges that keep twin groups whole, run one host thread and one pipeline per device with no
 * exchange between devices, and merge: the noise model's outputs are written in place by slot; the call lists of all
 * devices are copied to the first device (peer copies of exact sizes), sorted there into the reference's row order and
 * downloaded once.  Results are identical to a single-device context (tested).  _dev entry points, the element-wise
 * evaluators and as_fisher_tests_host run on devices[0].  The two programs use every visible GPU (AS_DEVICES=0,2,...
 * restricts them). */
int as_create_multi(const int* devices, int ndev, as_ctx** out);
/* The partition as_create_multi contexts use: n_shards contiguous, near-equal slot ranges [bounds_out[k], bounds_out[k+1])
 * (n_shards + 1 values), boundaries on multiples of 128 slots where possible, never inside a twin group (EE:1241-1245: all
 * slots of a position feed one estimate).  twin_next / twin_head may both be NULL.  Host arithmetic, no GPU needed. */
int as_shard_bounds(int64_t P, int32_t n_shards, const int32_t* twin_next, const int32_t* twin_head, int64_t* bounds_out);
/* Devices of a context: writes up to cap device ordinals, returns their number. */
int as_context_devices(const as_ctx* ctx, int* devices, int cap);
void as_destroy(as_ctx* ctx);
/* Pinned host memory for the _host entry points (cudaHostAlloc / cudaFreeHost). */
int as_host_alloc(void** out, size_t bytes);
int as_host_free(void* p);
/* Kernel variants (the tests cross-check them against each other and the oracle; -1 = default):
 *   caller: 0 = straightforward, 1 = per-warp queues over direct loads, TMA-staged with (samples per stage, stages):
 *           3 = (4,2), 11 = (3,2); with the integer pre-screen in the scan: 15 = (3,2), 14 = (4,2);
 *           13 = default: forward-first, the forward strand streamed (6,2) and a record's reverse-strand word fetched
 *           only when its forward strand can still make a call (single table; a sweep on 13 runs the deferred pipeline);
 *           20 = deferred: scan -> resolve -> series kernels over candidate lists (what a sweep of several tables runs)
 *   noise : 0 = direct loads; TMA-staged 1 = (4,3) default, 4 = (8,2), 6 = (4,2); 7, 8 = shared-pattern accumulators (the
 *           kernel of as_noise_estimate_sweep_dev) with the records of a stage interleaved / walked one by one */
int as_set_call_kernel(as_ctx* ctx, int variant);
int as_set_noise_kernel(as_ctx* ctx, int variant);
/* Slots per tile of the _host pipelines: 0 = automatic (~256 MiB of counts per buffer), else a multiple of 128.
 * Small values are for tests (tile-boundary handling). */
int as_set_host_tile_slots(as_ctx* ctx, int64_t slots);
/* Generic form of the setters above plus "deferred_capacity" (entries of the deferred caller's candidate list; 0 =
 * automatic; the kernels resolve what does not fit on the spot, so results never depend on it -- tests use tiny values)
 * and "forward_pending_cap" (usable entries of call kernel 13's per-control-warp ring of pending reverse-strand fetches,
 * 0 = automatic, at most 128; a full ring is drained on the spot, so results never depend on it either). */
int as_set_option(as_ctx* ctx, const char* name, int64_t value);
/* Number of kernel launches this context has enqueued so far (bench.py's gpu_launches). */
int64_t as_kernel_launches(const as_ctx* ctx);

/* ---- noise model: replaces storeGermlineStatistics (Germ_Max part, EE:1247-1467) and
 *      estimateThresholds (EE:1484-2544) ------------------------------------------------------
 * Inputs : counts of the S normals in the reference's file-iteration order (EE:1081; Germ_Max
 *          depends on it), twin_next/twin_head [P] or NULL, C = the float C_value (EE:329), cut >= 1.
 *          Slots [slot_begin, slot_end) of the tensor are processed; a twin group is processed when
 *          its head lies in the range (all of its members must be resident; they are written even when they
 *          lie outside the range).  The in-range members of a group whose head lies OUTSIDE the range are
 *          left unwritten: cut panels with as_shard_bounds, which never splits a group.
 * Outputs (per slot, indexed by slot; twins receive identical values):
 *   thr        float  [P][4][2]  fw,bw threshold per base; NaN = the "-1_-1" text (EE:1742-1770)
 *   germ_val   float  [P][4]     Germ_Max value: the maximal float(X)/float(RD) when germ_state == 2,
 *                                the floor (-888 for A, 0 for C,G,T; EE:1260, EE:1318) when 1
 *   germ_state uint8  [P][4]     0 = no entry ("-"), 1 = one qualifying record only, 2 = germ_val
 *   count      uint32 [P][4]     records that passed the filter (EE:1626)
 *   nrec       uint32 [P]        records of the position = Value_Hash.count() (EE:1742)          */
int as_noise_estimate_dev(as_ctx* ctx, const uint32_t* d_counts, int32_t S, int64_t P, int64_t slot_begin,
                          int64_t slot_end, const int32_t* d_twin_next, const int32_t* d_twin_head, float C,
                          int32_t cut, float* d_thr, float* d_germ_val, uint8_t* d_germ_state, uint32_t* d_count,
                          uint32_t* d_nrec, void* stream);
/* The _host forms also fill thr_view [P][4][2] when it is not NULL: the thresholds as the caller will parse them
 * (as_thresholds_caller_view_dev applied while the tile is still on the device). */
/* Noise-floor sweep (BASELINE configs[3]: C_value 0.001 ... 0.005): the noise model for n_c values of C in ONE pass over
 * the normals.  Only the sum of float(depth) * float(C) (EE:1617) depends on C; the filter, the depth and alt-read sums,
 * Germ_Max, count and nrec are shared, and the per-C sums are kept once per slot (not per base) for the records that carry
 * the slot's usual keep pattern (noise_pattern_kernel, as_noise_pattern.cu).  c_values is a HOST array [n_c],
 * 1 <= n_c <= 8; d_thr [n_c][P][4][2], table i = the thresholds as_noise_estimate_dev gives for c_values[i]
 * (bit-identical; tested).  The other outputs as in as_noise_estimate_dev. */
int as_noise_estimate_sweep_dev(as_ctx* ctx, const uint32_t* d_counts, int32_t S, int64_t P, int64_t slot_begin,
                                int64_t slot_end, const int32_t* d_twin_next, const int32_t* d_twin_head,
                                const float* c_values, int32_t n_c, int32_t cut, float* d_thr, float* d_germ_val,
                                uint8_t* d_germ_state, uint32_t* d_count, uint32_t* d_nrec, void* stream);
int as_noise_estimate_host(as_ctx* ctx, const uint32_t* counts, int32_t S, int64_t P, const int32_t* twin_next,
                           const int32_t* twin_head, float C, int32_t cut, float* thr, float* germ_val,
                           uint8_t* germ_state, uint32_t* count, uint32_t* nrec, float* thr_view);

/* The 16-bit wire format of the _host16 entry points: uint16 counts[sample][strand][slot][base], half the host footprint
 * and PCIe traffic of the uint32 layout.  A record whose eight counts are all < 65534 is stored as is; an absent record
 * is 0xFFFF in all eight words; a record with a larger count is ESCAPED -- 0xFFFE in all eight words -- and travels in
 * a side list of as_wide_record, sorted by slot.  Lossless for every input; the tile is widened to the uint32 layout on
 * the device, the kernels and results are the same. */
typedef struct {
    int32_t sample;
    int32_t slot;
    uint32_t fw[4];
    uint32_t bw[4];
} as_wide_record; /* 40 bytes */
#define AS_WIRE_ABSENT 0xFFFFu
#define AS_WIRE_ESCAPE 0xFFFEu
int as_noise_estimate_host16(as_ctx* ctx, const uint16_t* counts, const as_wide_record* wide, int64_t n_wide, int32_t S,
                             int64_t P, const int32_t* twin_next, const int32_t* twin_head, float C, int32_t cut, float* thr,
                             float* germ_val, uint8_t* germ_state, uint32_t* count, uint32_t* nrec, float* thr_view);

/* The packed wire format of the _host_packed entry points: uint32 packed[sample][strand][slot], ONE word per
 * (sample, strand, slot) = 8 bytes per record, a quarter of the uint32 layout.  A pileup row is one large count (the base
 * the sample carries) and three small ones (sequencing errors), so the word holds
 *     bits  0..15  the largest of the four counts ("major"; ties go to the lowest base index)
 *     bits 16..17  the base index of the major
 *     bits 18..21, 22..25, 26..29  the other three counts in ascending base order, each 0..15
 *     bits 30..31  zero
 * AS_PACKED_ABSENT in both strand words = no ASEQ row.  A record that does not fit (major > 65535 or another count > 15 on
 * either strand: germline / somatic variants, very noisy positions, ultra-deep coverage) is ESCAPED -- AS_PACKED_ESCAPE in
 * both words -- and travels in the side list of as_wide_record sorted by slot, exactly like the 16-bit format.  Lossless
 * for every input; the tile is unpacked to the uint32 layout on the device, kernels and results are the same.  Panels
 * where more than a few per cent of the records escape (e.g. 50,000x coverage) are better served by the 16-bit format. */
#define AS_PACKED_ABSENT 0xFFFFFFFFu
#define AS_PACKED_ESCAPE 0xFFFFFFFEu
/* Host helper: uint32 counts[n_samples][2][P][4] -> packed[n_samples][2][P] + wide records (sorted by slot, then sample).
 * *n_wide receives the number of escaped records; AS_EOVERFLOW when it exceeds wide_cap (call again with a larger list;
 * packed is complete either way).  Multi-threaded over samples; no GPU needed. */
int as_pack_counts(const uint32_t* counts, int32_t n_samples, int64_t P, uint32_t* packed, as_wide_record* wide,
                   int64_t wide_cap, int64_t* n_wide);
int as_noise_estimate_host_packed(as_ctx* ctx, const uint32_t* packed, const as_wide_record* wide, int64_t n_wide, int32_t S,
                                  int64_t P, const int32_t* twin_next, const int32_t* twin_head, float C, int32_t cut,
                                  float* thr, float* germ_val, uint8_t* germ_state, uint32_t* count, uint32_t* nrec,
                                  float* thr_view);

/* Noise-floor sweep on the _host path, in each of the three host formats (counts [+ wide, n_wide] as in the
 * single-value form): c_values is a host array [n_c], 1 <= n_c <= 8 (anything else: AS_EINVAL); thr and thr_view (when
 * not NULL) are [n_c][P][4][2].  Table i and its caller view are bit for bit what the single-value form returns for
 * c_values[i]; germ_val, germ_state, count and nrec (independent of C) are written once.  The counts go up once: each
 * upload tile runs noise_pattern_kernel for all values, the twin groups the tile holds once per value, and the twin
 * groups that straddle tiles are gathered once and reduced once per value.  n_c == 1 runs exactly the single-value
 * path (same kernels, same launches).  A multi-device context shards as the single-value forms do. */
int as_noise_estimate_sweep_host(as_ctx* ctx, const uint32_t* counts, int32_t S, int64_t P, const int32_t* twin_next,
                                 const int32_t* twin_head, const float* c_values, int32_t n_c, int32_t cut, float* thr,
                                 float* germ_val, uint8_t* germ_state, uint32_t* count, uint32_t* nrec, float* thr_view);
int as_noise_estimate_sweep_host16(as_ctx* ctx, const uint16_t* counts, const as_wide_record* wide, int64_t n_wide, int32_t S,
                                   int64_t P, const int32_t* twin_next, const int32_t* twin_head, const float* c_values,
                                   int32_t n_c, int32_t cut, float* thr, float* germ_val, uint8_t* germ_state, uint32_t* count,
                                   uint32_t* nrec, float* thr_view);
int as_noise_estimate_sweep_host_packed(as_ctx* ctx, const uint32_t* packed, const as_wide_record* wide, int64_t n_wide, int32_t S,
                                        int64_t P, const int32_t* twin_next, const int32_t* twin_head, const float* c_values,
                                        int32_t n_c, int32_t cut, float* thr, float* germ_val, uint8_t* germ_state,
                                        uint32_t* count, uint32_t* nrec, float* thr_view);

/* The noise table crosses to the caller as "%f" text (EE:1787 -> std::stof at VC:889-890) with
 * "-1_-1" replaced by "0.01_0.01" (EE:2680-2684).  This applies exactly that mapping to thr
 * [n] floats in place of the text round trip: NaN -> 0.01f, v -> strtof(sprintf("%f", v)). */
int as_thresholds_caller_view_dev(as_ctx* ctx, const float* d_thr, float* d_thr_view, int64_t n, void* stream);

/* ---- caller: replaces the row loop of callVariants (VC:723-3296: strand counts, threshold
 *      lookup, 3 alts x 2 strands of mutationRulesPoissonQualityScore VC:3834-3884 over the kfunc
 *      incomplete gamma VC:3720-3830, and the decision VC:898) --------------------------------
 * Inputs : tumour counts [T][2][P][4]; ref [P] (0..3, anything else = not callable, VC:3290);
 *          thr_view [P][4][2] = thresholds as the caller parsed them; cut >= 1.
 * Outputs: calls (unordered on the _dev path; sorted by (sample, slot, alt) = the reference's row
 *          order on the _host path), n_calls = true number found (the _dev path ADDS to
 *          *d_n_calls: zero it first).  Returns AS_EOVERFLOW when n_calls > cap (the first cap
 *          entries are valid).                                                                   */
int as_call_variants_dev(as_ctx* ctx, const uint32_t* d_counts, int32_t T, int64_t P, int64_t slot_begin,
                         int64_t slot_end, const uint8_t* d_ref, const float* d_thr_view, int32_t cut,
                         as_call* d_calls, int64_t cap, unsigned long long* d_n_calls, void* stream);
/* Noise-floor sweep (BASELINE configs[3]: C_value 0.001 ... 0.005): the caller for n_c threshold tables in ONE pass over
 * the tumour tensor.  d_thr_views [n_c][P][4][2] (table ci = the caller view of the noise model run with C_value ci),
 * d_calls [n_c][cap], d_n_calls [n_c] (zero them first).  The records are read once, the integer scan and its pre-screen
 * run once (against the smallest threshold of all tables), and only the candidates -- a few per thousand records --
 * are tested against every table.  List ci is what as_call_variants_dev returns for table ci (as a set; the lists are
 * unordered).  1 <= n_c <= 8; AS_EOVERFLOW semantics per list are the caller's to check (d_n_calls[ci] > cap). */
int as_call_variants_sweep_dev(as_ctx* ctx, const uint32_t* d_counts, int32_t T, int64_t P, int64_t slot_begin,
                               int64_t slot_end, const uint8_t* d_ref, const float* d_thr_views, int32_t n_c, int32_t cut,
                               as_call* d_calls, int64_t cap, unsigned long long* d_n_calls, void* stream);
int as_call_variants_host(as_ctx* ctx, const uint32_t* counts, int32_t T, int64_t P, const uint8_t* ref,
                          const float* thr_view, int32_t cut, as_call* calls, int64_t cap, int64_t* n_calls);

int as_call_variants_host16(as_ctx* ctx, const uint16_t* counts, const as_wide_record* wide, int64_t n_wide, int32_t T,
                            int64_t P, const uint8_t* ref, const float* thr_view, int32_t cut, as_call* calls, int64_t cap,
                            int64_t* n_calls);

int as_call_variants_host_packed(as_ctx* ctx, const uint32_t* packed, const as_wide_record* wide, int64_t n_wide, int32_t T,
                                 int64_t P, const uint8_t* ref, const float* thr_view, int32_t cut, as_call* calls,
                                 int64_t cap, int64_t* n_calls);

/* Caller sweep on the _host path, in each of the three host formats: thr_views [n_c][P][4][2], 1 <= n_c <= 8 (anything
 * else: AS_EINVAL), calls [n_c][cap], n_calls [n_c].  List i is what the single-table form returns for table i, in the same
 * order (sample, slot, alt); n_calls[i] is its true count.  AS_EOVERFLOW when any table has more than cap calls (the
 * first cap entries of every list are valid).  The tumour tensor goes up once; the n_c tables go up once ahead of the
 * first tile.  The kernel is chosen as as_call_variants_sweep_dev chooses it (the deferred pipeline by default, the
 * in-stage sweep kernel when a staged variant is selected); n_c == 1 runs exactly the single-table path.  Every table's
 * lists are sorted with one radix sort per table.  A multi-device context shards as the single-table forms do. */
int as_call_variants_sweep_host(as_ctx* ctx, const uint32_t* counts, int32_t T, int64_t P, const uint8_t* ref,
                                const float* thr_views, int32_t n_c, int32_t cut, as_call* calls, int64_t cap, int64_t* n_calls);
int as_call_variants_sweep_host16(as_ctx* ctx, const uint16_t* counts, const as_wide_record* wide, int64_t n_wide, int32_t T,
                                  int64_t P, const uint8_t* ref, const float* thr_views, int32_t n_c, int32_t cut, as_call* calls,
                                  int64_t cap, int64_t* n_calls);
int as_call_variants_sweep_host_packed(as_ctx* ctx, const uint32_t* packed, const as_wide_record* wide, int64_t n_wide, int32_t T,
                                       int64_t P, const uint8_t* ref, const float* thr_views, int32_t n_c, int32_t cut,
                                       as_call* calls, int64_t cap, int64_t* n_calls);

/* A device call list into the reference's row order (sample, slot, alt; VC:672, VC:723, VC:869-3288) without leaving the
 * device: slot_offset is added to every slot of d_calls first, IN PLACE (a shard's local slot ids -> panel slot ids), then one
 * radix sort of 64-bit keys and a row gather into d_sorted (n entries, must not overlap d_calls).  The final step of a multi-process run:
 * every rank's compacted list is sent to one rank (exact sizes), concatenated and sorted there (amplisolve_b200/shard.py). */
int as_sort_calls_dev(as_ctx* ctx, as_call* d_calls, int64_t n, int32_t slot_offset, as_call* d_sorted, void* stream);

/* ---- site report: the strand tests of listed SNVs in every tumour, called or not -------------------------------------
 * The reference evaluates mutationRulesPoissonQualityScore (VC:3834-3884, over the kfunc incomplete gamma VC:3720-3830 with
 * both branches and their 99-step caps) for both strands of every row and alt (VC:895-896) and applies the decision of VC:898
 * afterwards; the caller entry points above keep only the calls.  These entry points keep every test of the listed sites:
 * site i is (site_slot[i], site_alt[i]), and for every table c and tumour t, out[(c * T + t) * n_sites + i] holds the record's
 * strand depths (the sums of the four counts, VC:760-770), the alt reads, p_fw / p_bw = the double p of VC:3858-3866 on the
 * caller view of table c (1 when k = 0; no screen: the p of every present, testable record, whatever its coverage) and one
 * of the statuses below.  AS_SITE_CALLED is exactly the decision of the caller entry points (same device arithmetic):
 * present, FW >= cut and BW >= cut, ref in 0..3, alt != ref and both strands reach Q >= 5.
 * p is NaN where it is not evaluated (NO_DATA, NOT_TESTABLE, and a threshold of -1, whose Q is the reference's -888); the
 * counts of a NO_DATA entry are 0. */
#define AS_SITE_CALLED 1       /* the caller calls (tumour, slot, alt) with this table */
#define AS_SITE_NOT_CALLED 2   /* present and covered; a strand's Q is below 5 */
#define AS_SITE_LOW_COVERAGE 3 /* present, FW < cut or BW < cut (VC:898); p is still evaluated */
#define AS_SITE_NO_DATA 4      /* the record is absent (no ASEQ row) */
#define AS_SITE_NOT_TESTABLE 5 /* the slot's reference base is not A/C/G/T (VC:3290-3293), or alt = ref */
typedef struct {
    uint32_t depth_fw, depth_bw; /* FW, BW of VC:760-770 */
    uint32_t alt_fw, alt_bw;     /* alt reads per strand */
    double p_fw, p_bw;           /* VC:3858-3866 per strand (VC:895-896) */
    int32_t status;              /* AS_SITE_* */
    int32_t pad;
} as_site_test; /* 40 bytes */
/* counts [T][2][P][4] (+ wide, n_wide) in any of the three host formats, ref [P] and thr_views [n_c][P][4][2] exactly as
 * as_call_variants_sweep_host* take them; site_slot / site_alt [n_sites]; out [n_c][T][n_sites].  1 <= n_c <= 8, every
 * slot in [0, P) and every alt in 0..3, else AS_EINVAL; n_sites = 0 or T = 0 return AS_OK with nothing written.  The host
 * gathers the sites' columns of counts in their format (escaped records follow, renumbered by site) and uploads them as a
 * count tensor of n_sites slots, which the wire-format path widens on the device; site_test_kernel (as_sites.cu) then
 * evaluates every (table, site, tumour, strand).  A multi-device context runs this on its first device: the work is the
 * sites' columns, not the panel. */
int as_site_tests_host(as_ctx* ctx, const uint32_t* counts, int32_t T, int64_t P, const uint8_t* ref, const float* thr_views,
                       int32_t n_c, const int32_t* site_slot, const int32_t* site_alt, int64_t n_sites, int32_t cut,
                       as_site_test* out);
int as_site_tests_host16(as_ctx* ctx, const uint16_t* counts, const as_wide_record* wide, int64_t n_wide, int32_t T, int64_t P,
                         const uint8_t* ref, const float* thr_views, int32_t n_c, const int32_t* site_slot, const int32_t* site_alt,
                         int64_t n_sites, int32_t cut, as_site_test* out);
int as_site_tests_host_packed(as_ctx* ctx, const uint32_t* packed, const as_wide_record* wide, int64_t n_wide, int32_t T, int64_t P,
                              const uint8_t* ref, const float* thr_views, int32_t n_c, const int32_t* site_slot,
                              const int32_t* site_alt, int64_t n_sites, int32_t cut, as_site_test* out);

/* Element-wise Poisson test on the device: p[i] = the double p-value of VC:3858-3866 and
 * q[i] = the Q score of VC:3868-3882 for (k[i], rd[i], err[i]).  Host pointers.  Used by the
 * parity tests to compare the device incomplete gamma with the reference's on arbitrary grids. */
int as_poisson_test_host(as_ctx* ctx, const int32_t* k, const int32_t* rd, const float* err, int64_t n, double* p,
                         double* q);
/* kf_gammaq(s, z) of VC:3726 evaluated on the device, element-wise.  Host pointers. */
int as_kf_gammaq_host(as_ctx* ctx, const double* s, const double* z, int64_t n, double* out);

/* ---- synthetic count tensors generated directly in HBM (benchmark inputs; SURVEY.md 8d) ------
 * Fills d_counts [n_samples][2][P][4] with the seeded synthetic panel model: log-normal depth,
 * per-slot strand-specific error rates, germline SNPs, spiked somatic SNVs (tumours only) and
 * absent rows.  d_ref [P] receives the reference base of each slot when non-NULL. */
typedef struct {
    uint64_t seed;
    float mean_depth;     /* e.g. 2000 */
    float depth_sigma;    /* log-normal sigma of per-(sample,slot) depth, e.g. 0.5 */
    float germline_rate;  /* fraction of slots carrying a germline SNP, e.g. 1e-3 */
    float somatic_rate;   /* spiked SNVs per (sample,slot); 0 for normals */
    float somatic_vaf_lo; /* e.g. 0.01 */
    float somatic_vaf_hi; /* e.g. 0.2 */
    float absent_rate;    /* fraction of (sample,slot) records dropped */
    int32_t sample_offset; /* global index of the first sample (decorrelates normals and tumours) */
    int64_t slot_offset;   /* global index of the first slot (position sharding across GPUs); multiple of 125 */
    int32_t twin_period;   /* 0 = no duplicated positions; n = one amplicon junction in n overlaps by 2..10 positions */
    int32_t reserved;
} as_synth_params;
int as_synth_counts_dev(as_ctx* ctx, uint32_t* d_counts, int32_t n_samples, int64_t P, uint8_t* d_ref,
                        const as_synth_params* prm, void* stream);
/* twin_next / twin_head [P] of the synthetic panel geometry (125-slot amplicons, see twin_period). */
int as_synth_twin_links_dev(as_ctx* ctx, int64_t P, const as_synth_params* prm, int32_t* d_twin_next,
                            int32_t* d_twin_head, void* stream);

/* ---- pileup: BAM records -> the count tensor of one sample (SURVEY.md 8 f4) ---------------------
 * Replaces the pre-processing step of the reference, `./ASEQ vcf= bam= mbq= mrq= mdc= out=` alias computeCounts
 * (Execution_examples.md:16-54; the reference ships it as a binary only, so this is a new design with the conventions of
 * a samtools-style pileup -- amplisolve_b200/csrc/as_pileup.cu states them -- and its parity with that binary is unpinned).
 * The panel is given as the sorted, unique, 0-based positions of each contig: slot_pos[contig_first[c] .. contig_first[c+1]).
 * as_pileup_begin   uploads the panel and zeroes the device counts [2 strands][P][4 bases];
 * as_pileup_add_host adds the reads of a piece of the UNCOMPRESSED record stream of a BAM file (header stripped):
 *                   records[0..n_bytes), rec_off[i] = byte offset of record i (its block_size field), ref_contig[refID] =
 *                   panel contig of a BAM reference sequence or -1.  A read counts when mapq >= mrq and (flag & skip_flags)
 *                   == 0; a base when it is aligned (M, =, X), A/C/G/T and of quality >= mbq.  Any number of pieces.
 * as_pileup_end_host downloads counts (host, 2 * P * 4 uint32: forward strand first) and the number of reads / bases
 *                   used (stats_out[2], may be NULL).
 * The device buffer keeps the layout of one sample of the count tensor, [strand][slot][base].
 * How a BAM file yields the count tensor of the two programs (a germline_dir= / tumour_dir= that holds *.bam files and no
 * *.ASEQ file): the P slots of the program's panel map to the U sorted unique positions of the pileup through
 * slot_unique[P] (twin slots name the same position); the pileup of each BAM runs on the GPU and ends with
 * as_pileup_end_wire instead of as_pileup_end_host, which writes that sample's slice of the host wire tensor directly:
 * slot s gets the record of position slot_unique[s], or is ABSENT when the depth of that record (the sum of its eight
 * counts, in 64 bits) is below mdc.  The result is the tensor the ASEQ loader builds from the files computeCounts writes
 * with the same mbq / mrq / mdc for a position file that lists the panel's slots in order.
 * as_pileup_end_wire: fmt 1 = packed, wire = uint32 [2][P] (forward words first, then reverse); fmt 2 = 16-bit, wire =
 *                   uint16 [2][P][4]; ABSENT / ESCAPE markers as above.  Escaped records go to wide (sample = `sample`,
 *                   sorted by slot); *n_wide = their number, AS_EOVERFLOW when it exceeds wide_cap (wire and *n_wide are
 *                   complete; the pileup stays open, so the call can be repeated with a larger list).  *rows_out = present
 *                   slots, stats_out[2] as in as_pileup_end_host (both may be NULL).  AS_EINVAL for a slot_unique entry
 *                   outside [0, U).  Ends the pileup on success.
 * as_pileup_set_host replaces the counts of the open pileup with host counts [2][U][4] (a pileup made elsewhere; tests).
 * A context of several GPUs runs the pileup on its first. */
int as_pileup_begin(as_ctx* ctx, const int64_t* contig_first, int32_t n_contig, const int32_t* slot_pos, int64_t P);
int as_pileup_add_host(as_ctx* ctx, const uint8_t* records, int64_t n_bytes, const int64_t* rec_off, int64_t n_rec,
                       const int32_t* ref_contig, int32_t n_ref, int32_t mbq, int32_t mrq, uint32_t skip_flags);
int as_pileup_end_host(as_ctx* ctx, uint32_t* counts, uint64_t* stats_out);
int as_pileup_end_wire(as_ctx* ctx, const int32_t* slot_unique, int64_t P, int32_t mdc, int32_t fmt, int32_t sample, void* wire,
                       as_wide_record* wide, int64_t wide_cap, int64_t* n_wide, int64_t* rows_out, uint64_t* stats_out);
int as_pileup_set_host(as_ctx* ctx, const uint32_t* counts);

/* ---- host side of the two programs (text formats; amplisolve_b200/csrc/as_host.cpp) ---------- */
/* Iteration order of a libstdc++ std::unordered_map<std::string,std::string> after inserting keys
 * in the given sequence: the order in which the reference walks its file lists (EE:1081, VC:672).
 * order_out[i] = index into keys of the i-th visited entry.  Returns the number of entries. */
int as_hash_iteration_order(const char* const* keys, int32_t n, int32_t* order_out);

/* Two-sided Fisher exact test of strand bias, fisherTest(a = RD_fw, b = RD_bw, c = alt reads fw, d = alt reads bw) of
 * VC:3797-3814, as as_variant_calling_main evaluates it for every call (VC:902): cutoff = pdf(c) of the hypergeometric
 * distribution (r = a + c, n = c + d, N = a + b + c + d), p = sum of the pdf(k) <= cutoff over k ascending.  The reference
 * takes pdf from Boost.Math 1.61 (not in its tree); here pdf is C(r,k) C(N-r,n-k) / C(N,n) through lgamma.  Host code, no
 * GPU needed.  Returns -1 for a negative argument. */
double as_fisher_test(int32_t fw, int32_t bw, int32_t alt_fw, int32_t alt_bw);

/* The same test for n tables at once on the device (SURVEY.md 8 f3): tables [n][4] = {fw, bw, alt_fw, alt_bw}, p [n].
 * One warp per table, lanes over the support of the hypergeometric distribution; the log-domain terms come from a
 * lgamma table filled by the host (bit-identical to as_fisher_test), exp is the device's, the partial sums of the 32
 * lanes are added in ascending k: p agrees with as_fisher_test to a few ulp (tests: <= 1e-13 relative, identical
 * printed strings and YES/NO flags).  Tables whose N = fw + bw + alt_fw + alt_bw exceeds 2^26 are evaluated on the host.
 * Host pointers.  as_variant_calling_main uses this for the FisherPvalue column. */
int as_fisher_tests_host(as_ctx* ctx, const int32_t* tables, int64_t n, double* p);

/* Whole programs, argv-compatible with the reference (EE:241-520, VC:199-360).  Exit status is
 * the return value; like the reference, usage errors print the usage text and return 0.  germline_dir= / tumour_dir= may
 * also name a directory of *.bam files (and no *.ASEQ file): the programs then pile the BAMs up on the GPU themselves, with
 * mbq / mrq / mdc from AS_BAM_MBQ / AS_BAM_MRQ / AS_BAM_MDC (default 20 / 20 / 20, skip flags 0x704), and write what
 * computeCounts followed by the same program would write. */
int as_error_estimation_main(int argc, char** argv);
int as_variant_calling_main(int argc, char** argv);
/* computeCounts / ASEQ PILEUP mode (Execution_examples.md:27): [vcf=positions] [bam=file.bam] [threads=n] [mbq=n] [mrq=n]
 * [mdc=n] [out=dir] -> <out>/<bam name>.PILEUP.ASEQ, the 15-column text both programs above read.  BGZF blocks are
 * inflated on `threads` host threads, the pileup runs on the GPU (as_pileup_*). */
int as_compute_counts_main(int argc, char** argv);

/* ---- resident service (amplisolve_b200/csrc/as_serve.cpp; no counterpart in the reference) -----
 * A CUDA process pays 0.25 - 5 s for its context before the first kernel; the three programs above do a few tenths of a
 * second of work on a gene panel.  as_serve_main (`amplisolve_b200_serve socket=<path> [devices=0,1]`) keeps a context
 * open and runs the programs of clients in its own process; as_client_run is what the thin mains call first: with
 * AS_SERVER=<path> in the environment and a service listening it ships argv, the working directory, the AS_* environment
 * and the caller's stdout / stderr descriptors, waits, stores the exit status in *rc_out and returns 1; otherwise it
 * returns 0 and the caller runs as_*_main itself.  prog: 0 error estimation, 1 variant calling, 2 compute counts.
 * as_process_is_resident: 1 inside the service (a program's context is then destroyed when it returns). */
int as_serve_main(int argc, char** argv);
int as_client_run(int prog, int argc, char** argv, int* rc_out);
int as_process_is_resident(void);

#ifdef __cplusplus
}
#endif
#endif /* AMPLISOLVE_B200_H */
