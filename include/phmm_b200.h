/*
 * phmm_b200.h — C ABI of the B200-native pair-HMM haplotype-likelihood engine.
 *
 * Drop-in boundary for ONE path of luntergroup/octopus (v0.7.4): the banded pair-HMM that scores every
 * (read, haplotype) pair and fills HaplotypeLikelihoodArray. The reference has no FFI layer; the seams this
 * ABI replaces are (paths relative to the reference tree):
 *
 *   raw kernel    simd::PairHMM::align(truth, target, quals, truth_len, target_len, snv_mask, snv_prior,
 *                 gap_open, gap_extend, nuc_prior)            src/core/models/pairhmm/simd_pair_hmm.hpp:454-470
 *                 → phmm_align_scores()           (one integer score per (read, haplotype window) task)
 *   per read      hmm::evaluate(truth, target, quals, offset, hmm, params)      pair_hmm.hpp:827-841
 *                 HaplotypeLikelihoodModel::evaluate(read, first_pos, last_pos) haplotype_likelihood_model.cpp:261-304
 *   batch         HaplotypeLikelihoodArray::populate(reads, haplotypes, flank_state, workers)
 *                                                              haplotype_likelihood_array.cpp:51-103
 *                 → phmm_populate()               (the [H][R] matrix of ln-likelihoods, double)
 *
 * Conventions: plain pointers and sizes only; every pointer of one call lives in the memory space named by
 * `space` (host memory, or device memory of the engine's GPU); the caller owns all buffers; calls are
 * synchronous (results complete on return) unless stated; functions return PHMM_OK or a negative error code
 * and never throw — the C++ adapter (octopus_b200/cpp/phmm_b200.hpp) re-throws the reference's exceptions.
 * An engine handle is not re-entrant (one per host thread, like the reference's per-thread model copies,
 * haplotype_likelihood_array.cpp:172).
 * There is no CPU fallback: every entry point that computes fails with PHMM_ERR_CUDA when no B200 is usable.
 */
#ifndef PHMM_B200_H
#define PHMM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHMM_OK                  0
#define PHMM_ERR_INVALID        -1   /* bad argument (message in phmm_last_error) */
#define PHMM_ERR_CUDA           -2   /* CUDA runtime / no device */
#define PHMM_ERR_BAND           -3   /* band > 256: reference TooLargeBandSizeError (simd_pair_hmm_wrapper.hpp:45-61) */
#define PHMM_ERR_SHORT_HAPLOTYPE -4  /* reference ShortHaplotypeError (haplotype_likelihood_model.cpp:238-256); see status[] */
#define PHMM_ERR_NOMEM          -5

#define PHMM_SPACE_HOST   0
#define PHMM_SPACE_DEVICE 1

/* per-pair status written by phmm_populate (optional output) */
#define PHMM_STATUS_OK          0
#define PHMM_STATUS_OVERFLOW    1   /* every candidate returned lowest(): pair_hmm.hpp:736-738,750-752 */
#define PHMM_STATUS_SHORT_HAP   2   /* ShortHaplotypeError; required extension in the high 16 bits */

typedef struct phmm_engine phmm_engine;

/* mirrors HaplotypeLikelihoodModel::Config (haplotype_likelihood_model.hpp:36-44) + hmm::Parameters::nuc_prior */
typedef struct {
    int32_t max_indel_error;             /* requested band; rounded up to 8,16,32,...,256 (simd_pair_hmm_wrapper.hpp:218-241) */
    int32_t use_int_scores;              /* reference: int32 SIMD lanes. Here: forces the 32-bit kernel */
    int32_t use_mapping_quality;         /* default 1 */
    int32_t mapping_quality_cap;         /* default 120 */
    int32_t mapping_quality_cap_trigger; /* < 0: none (boost::none) */
    int32_t use_flank_state;             /* default 1 */
    int32_t nuc_prior;                   /* default 2 (pair_hmm.hpp:86) */
    int32_t disable_naive_shortcut;      /* 1: every candidate goes through the DP (benchmark mode; NOT reference behaviour) */
    int32_t map_positions;               /* 1 (default): when no candidate positions are supplied, compute them on the device with
                                            the reference's k-mer mapper (utils/kmer_mapper.hpp:43-159, K = 6, <= 10 positions), as
                                            populate does inline (haplotype_likelihood_array.cpp:89-92); 0: original position only */
} phmm_config;

/* H haplotypes, struct of arrays. Per-base arrays are concatenated; haplotype h owns [off[h], off[h+1]).
 * These are exactly the members HaplotypeLikelihoodModel::reset fills (haplotype_likelihood_model.cpp:60-78). */
typedef struct {
    int32_t        n;
    const int64_t* off;            /* [n+1] */
    const char*    seq;            /* Haplotype::sequence() */
    const char*    snv_mask_fwd;   /* haplotype_snv_forward_mask_ */
    const int8_t*  snv_prior_fwd;  /* haplotype_snv_forward_priors_ */
    const char*    snv_mask_rev;
    const int8_t*  snv_prior_rev;
    const int8_t*  gap_open;       /* haplotype_gap_open_penalities_ */
    const int8_t*  gap_extend;     /* haplotype_gap_extend_penalities_ */
    const int64_t* begin;          /* [n] mapped_begin(haplotype), or NULL (= 0) */
} phmm_haplotypes;

/* R reads, struct of arrays (AlignedRead fields: basics/aligned_read.hpp:36-39,120-146). */
typedef struct {
    int32_t        n;
    const int64_t* off;            /* [n+1] */
    const char*    bases;          /* AlignedRead::sequence() */
    const uint8_t* quals;          /* AlignedRead::base_qualities() */
    const uint8_t* mapq;           /* [n] AlignedRead::mapping_quality() */
    const uint8_t* reverse;        /* [n] AlignedRead::is_marked_reverse_mapped() */
    const int64_t* begin;          /* [n] mapped_begin(read): original position = begin[r] - haplotype begin[h] */
} phmm_reads;

/* Candidate mapping positions per (haplotype, read) pair, CSR in [H][R] order
 * (what map_query_to_target emits, utils/kmer_mapper.hpp:120-159). NULL → mapped on the device (config.map_positions = 1)
 * or only the original position is tried (map_positions = 0). */
typedef struct {
    const int64_t* off;            /* [H*R + 1] */
    const int32_t* pos;
} phmm_positions;

/* HaplotypeLikelihoodModel::FlankState (haplotype_likelihood_model.hpp:46-49); has_flank = 0 ↔ boost::none */
typedef struct {
    int32_t has_flank;
    int64_t lhs_flank, rhs_flank;
} phmm_flank_state;

/* One raw-kernel task: read `read` against the window of haplotype `hap` starting at `win_off`
 * (window length = read length + 2*band - 1), SNV mask/prior of strand `reverse`. */
typedef struct {
    int32_t read;
    int32_t hap;
    int32_t win_off;
    int32_t reverse;
} phmm_task;

/* One (read, haplotype) pair of phmm_align_reads. */
typedef struct {
    int32_t read;
    int32_t hap;
} phmm_pair;

#define PHMM_STATUS_CIGAR_TRUNCATED 3   /* phmm_align_reads: cigar_stride too small */
#define PHMM_STATUS_HMM_OVERFLOW    4   /* reference HMMOverflow (pair_hmm.hpp:47-64, 815-817) */

const char* phmm_version(void);
void        phmm_default_config(phmm_config* cfg);

/* device < 0: current CUDA device. Creates the engine's stream and scratch pools. */
int         phmm_create(phmm_engine** out, int device);
void        phmm_destroy(phmm_engine* e);
const char* phmm_last_error(const phmm_engine* e);   /* valid until the next call on e; e may be NULL */

/* Stream ordering (SURVEY.md §8b: "synchronous unless a stream handle is passed"). Calls run on the engine's own non-blocking CUDA
 * stream and are complete when they return, which orders them after everything the HOST has waited for. Work the caller has
 * merely ENQUEUED on another stream — e.g. an NCCL gather still reading the buffer the next call will overwrite — is ordered by
 * handing the engine an event recorded after that work: phmm_wait_event(e, ev) makes the engine's stream(s) wait for `ev`
 * (a cudaEvent_t) on the device before anything enqueued by later calls runs. phmm_engine_stream returns the engine's cudaStream_t
 * for callers that want to record or wait on it themselves. */
int         phmm_wait_event(phmm_engine* e, void* cuda_event);
void*       phmm_engine_stream(phmm_engine* e);
/* The persistent DP kernels occupy every SM; a collective the caller runs BESIDE the next call (the gather of the previous result) then
 * waits for them. n_sms > 0 keeps the first n_sms SMs free of DP blocks (cost: n_sms / 148 of the DP throughput); 0 (default) = none. */
int         phmm_reserve_sms(phmm_engine* e, int n_sms);

/* Page-locked host memory (cudaHostAlloc) for callers that do not link the CUDA runtime themselves: host-space calls on pinned
 * buffers copy at full rate and overlap with compute. NULL when no GPU / out of memory (callers fall back to malloc). */
void*       phmm_host_alloc(size_t bytes);
void        phmm_host_free(void* p);

/* Number of kernels of this library launched by the last call / in total (bench.py's gpu_launches). */
int64_t     phmm_launch_count(const phmm_engine* e, int total);

/* CUDA events around the dominant DP kernel of the last call, in milliseconds (0 if none ran). */
double      phmm_last_dp_kernel_ms(const phmm_engine* e);
/* Banded cells 2*(L+band)*band summed over the DP tasks of the last call (the GCUPS numerator, SURVEY §8d). */
int64_t     phmm_last_dp_cells(const phmm_engine* e);

/* Raw kernel boundary: scores[j] == reference hmm.align(hap window, read, ...) for task j (integer phred).
 * band must be one of 8,16,32,...,256. precision_bits: 16 (packed s16x2 fast path where it is exact, else 32) or 32. */
int phmm_align_scores(phmm_engine* e, int band, int precision_bits, int nuc_prior,
                      const phmm_haplotypes* haps, const phmm_reads* reads,
                      const phmm_task* tasks, int64_t n_tasks, int32_t* scores, int space);

/* Per-call seam with traceback, host pointers only: the reference kernel's traceback overload
 *   hmm.align(truth, target, quals, truth_len, target_len, snv_mask, snv_prior, gap_open, gap_extend, nuc_prior,
 *             first_pos, align1, align2)                                   simd_pair_hmm.hpp:491-509
 * truth_len must be target_len + 2*band - 1; snv_mask == NULL selects the no-SNV overload (:472-489) and
 * gap_extend == NULL the scalar-extend overload (value gap_extend_scalar). align1 / align2: caller-allocated,
 * >= 2*(target_len + band) + 1 bytes, NUL-terminated on return ('-' marks gaps); *first_pos = -1 on overflow. */
int phmm_align_traceback(phmm_engine* e, int band,
                         const char* truth, const char* target, const int8_t* quals, int truth_len, int target_len,
                         const char* snv_mask, const int8_t* snv_prior, const int8_t* gap_open,
                         const int8_t* gap_extend, int gap_extend_scalar, int nuc_prior,
                         int* score, int* first_pos, char* align1, char* align2);

/* Best alignment of explicit (read, haplotype) pairs: HaplotypeLikelihoodModel::align (haplotype_likelihood_model.cpp:397-431 →
 * compute_optimal_alignment :335-395 → hmm::align pair_hmm.hpp:858-874), the call ReadRealigner / ReadAssigner make
 * (core/tools/read_realigner.cpp:100-150). positions: CSR over the PAIR LIST (off[n_pairs+1]) or NULL.
 * Outputs per pair: mapping_position (Alignment::mapping_position), likelihood (after mapping-quality mixing), the CIGAR as
 * text with the reference's operation letters (= X I D; basics/cigar_string.hpp:27-31) in cigar[j*cigar_stride ..),
 * status[j] (PHMM_STATUS_*; SHORT_HAP / HMM_OVERFLOW correspond to the reference's exceptions). */
int phmm_align_reads(phmm_engine* e, const phmm_config* cfg,
                     const phmm_haplotypes* haps, const phmm_reads* reads,
                     const phmm_pair* pairs, int64_t n_pairs,
                     const phmm_positions* positions, const phmm_flank_state* flank,
                     int64_t* mapping_position, double* likelihood, char* cigar, int32_t cigar_stride, int32_t* status, int space);

/* hmm::align itself, batched (pair_hmm.hpp:858-874 → try_naive_align :321-340, simd_align :784-823): pair j aligns target
 * `pairs[j].read` of the `targets` block against truth `pairs[j].hap` of the `truths` block at target offset target_offsets[j] — no
 * candidate enumeration, no in-range rule. This is the call DeNovoModel makes per (haplotype, haplotype) pair
 * (core/models/mutation/denovo_model.cpp:249-290: PairHMM<VariableGapExtendMutationModel, 32, int>::align(target, padded given)) and
 * haplotype_filter's likelihood ranking builds on: pack the padded "given" haplotypes as truths (gap_open / gap_extend arrays; an SNV mask
 * that matches no base, e.g. 0 bytes, is the no-SNV overload), the "target" haplotypes as targets with every quality = the model's
 * scalar mismatch penalty (pair_hmm.hpp:853-856), max_indel_error = 32, use_mapping_quality = 0, offset = the band.
 * Outputs per pair as phmm_align_reads: Alignment::target_offset, likelihood (-ln10/10 * score), CIGAR text; a window that does not fit
 * gives {0, lowest(), ""} (:802-807); status PHMM_STATUS_HMM_OVERFLOW ↔ HMMOverflow. targets->mapq may be NULL when use_mapping_quality = 0. */
int phmm_align_pairs(phmm_engine* e, const phmm_config* cfg,
                     const phmm_haplotypes* truths, const phmm_reads* targets,
                     const phmm_pair* pairs, const int32_t* target_offsets, int64_t n_pairs, const phmm_flank_state* flank,
                     int64_t* target_offset_out, double* likelihood, char* cigar, int32_t cigar_stride, int32_t* status, int space);

/* Batch boundary: out[h*R + r] == HaplotypeLikelihoodArray likelihoods_[h][sample][r] for a single-sample ReadMap
 * (haplotype_likelihood_array.cpp:77-95). status (optional, [H*R]) receives PHMM_STATUS_*.
 * Returns PHMM_ERR_SHORT_HAPLOTYPE if any pair raised ShortHaplotypeError (the reference throws out of populate). */
int phmm_populate(phmm_engine* e, const phmm_config* cfg,
                  const phmm_haplotypes* haps, const phmm_reads* reads,
                  const phmm_positions* positions, const phmm_flank_state* flank,
                  double* out, int32_t* status, int space);

/* Many regions in one call. Octopus runs populate once per ACTIVE REGION (Caller::call_variants, core/callers/caller.cpp:445-531 →
 * compute_haplotype_likelihoods :1159-1196): a few to a few hundred haplotypes x some hundred to some thousand reads — far too small
 * to fill a B200 (one such call is launch-latency bound). Here region g owns the haplotypes [hap_first[g], hap_first[g+1]) and the
 * reads [read_first[g], read_first[g+1]) of the two blocks; every read is scored against the haplotypes of its own region only, all
 * regions in ONE kernel chain. The region arrays live in HOST memory whatever `space` says (they are tiny and the host sizes the
 * call from them). */
typedef struct {
    int32_t                 n;            /* regions */
    const int32_t*          hap_first;    /* [n+1], hap_first[0] = 0, hap_first[n] = haplotypes->n */
    const int32_t*          read_first;   /* [n+1] likewise over the reads */
    const phmm_flank_state* flank;        /* [n] per-region flank state, or NULL (none) */
} phmm_regions;

/* out / status (optional): the regions' row-major [H_g][R_g] matrices back to back, region g starting at sum_{g' < g} H_g' * R_g'.
 * Candidate positions come from the device k-mer mapper (config.map_positions) or are the original position only. Errors and statuses
 * as phmm_populate. At most 65535 haplotypes per call. This is phmm_populate_regions_ex(e, cfg, haps, reads, regions, NULL, NULL, out,
 * status, space); that call adds paired-read templates and explicit candidate positions. */
int phmm_populate_regions(phmm_engine* e, const phmm_config* cfg,
                          const phmm_haplotypes* haps, const phmm_reads* reads, const phmm_regions* regions,
                          double* out, int32_t* status, int space);

/* Templates of a many-regions call. Region g owns the templates [template_first[g], template_first[g+1]).
 * Template t owns the reads [template_off[t], template_off[t+1]); each region's templates cover exactly its reads. */
typedef struct {
    const int32_t* template_first;   /* [regions->n + 1], HOST memory whatever `space` says (like the region arrays) */
    const int64_t* template_off;     /* [template_first[n] + 1], in `space` */
} phmm_region_templates;

/* Many regions in one call with Octopus's default read linkage: populate(TemplateMap) per region (haplotype_likelihood_array.cpp:105-199,
 * caller.cpp:465-468) — the value of a template is the sum of its reads' values, in read order (haplotype_likelihood_model.cpp:306-320).
 *   templates  NULL: one value per read, as phmm_populate_regions. Otherwise out holds the regions' [H_g][T_g] matrices back to back.
 *              A sample of a multi-sample region is a column range: put the samples' templates back to back.
 *   positions  NULL: device mapper / original position, as phmm_populate_regions. Otherwise a CSR over the per-read result slots
 *              (off[sum_g H_g * R_g + 1], the [H_g][R_g] layout of status), validated as in phmm_populate (<= 4096 per pair).
 *   status     optional, always per read: the regions' [H_g][R_g] matrices back to back.
 * Template offsets in host memory are checked on the host, device ones on the device; either way a malformed list (not non-decreasing,
 * or a region's templates not covering exactly its reads) returns PHMM_ERR_INVALID. A short haplotype in one region returns
 * PHMM_ERR_SHORT_HAPLOTYPE with the statuses and values of every region complete (the caller skips that region, caller.cpp:1182-1188). */
int phmm_populate_regions_ex(phmm_engine* e, const phmm_config* cfg,
                             const phmm_haplotypes* haps, const phmm_reads* reads, const phmm_regions* regions,
                             const phmm_region_templates* templates, const phmm_positions* positions,
                             double* out, int32_t* status, int space);

/* phmm_populate with device-resident inputs and an output row stride: out[h * out_ld + r], out_ld >= R (status, optional, stays dense
 * [H][R]). `out` is any device-accessible address — in particular a window of ANOTHER GPU's matrix mapped with phmm_ipc_open: the
 * epilogue kernel then stores this rank's columns of a read-sharded [H, R_total] matrix (or its slab of a per-rank stack) straight
 * into the owner's HBM over NVLink / NVSwitch, and no gather collective follows (DESIGN.md section 7). */
int phmm_populate_ld(phmm_engine* e, const phmm_config* cfg,
                     const phmm_haplotypes* haps, const phmm_reads* reads,
                     const phmm_positions* positions, const phmm_flank_state* flank,
                     double* out, int64_t out_ld, int32_t* status);

/* Peer output memory (one node, one process per GPU). The owner allocates the result matrix with phmm_device_alloc (cudaMalloc, the
 * allocation CUDA IPC can export), exports it once, and sends the 64 handle bytes to the other processes by any means; they map it
 * with phmm_ipc_open (peer access is enabled on demand) and pass addresses inside it to phmm_populate_ld. A writer's stores are
 * complete when its call has returned; the owner learns that through the caller's own barrier. phmm_ipc_close unmaps. */
#define PHMM_IPC_HANDLE_BYTES 64
int phmm_device_alloc(int device, size_t bytes, void** dev_ptr);
int phmm_device_free(void* dev_ptr);
int phmm_ipc_export(const void* dev_ptr, unsigned char handle[PHMM_IPC_HANDLE_BYTES]);
int phmm_ipc_open(int device, const unsigned char handle[PHMM_IPC_HANDLE_BYTES], void** dev_ptr);
int phmm_ipc_close(void* dev_ptr);

/* Paired / linked reads: HaplotypeLikelihoodArray::populate(TemplateMap) (haplotype_likelihood_array.cpp:105-199). Template t owns
 * the reads [template_off[t], template_off[t+1]) and its value is the sum of its reads' values
 * (HaplotypeLikelihoodModel::evaluate(AlignedTemplate), haplotype_likelihood_model.cpp:306-320). out is [H][n_templates];
 * status (optional) stays per read, [H][R]. Everything else as phmm_populate. The one-region case of phmm_populate_regions_ex. */
int phmm_populate_templates(phmm_engine* e, const phmm_config* cfg,
                            const phmm_haplotypes* haps, const phmm_reads* reads,
                            const int64_t* template_off, int32_t n_templates,
                            const phmm_positions* positions, const phmm_flank_state* flank,
                            double* out, int32_t* status, int space);

/* Consumer of the matrix ("next" row N1): ConstantMixtureGenotypeLikelihoodModel::evaluate for G genotypes of one ploidy
 * (core/models/genotype/constant_mixture_genotype_likelihood_model.cpp:30-140) over a [H][R] matrix in `space`:
 *   out[g] = sum_r ( log_sum_exp_{h in genotype g} lnl[h*R + r] - ln ploidy ),   genotypes[g*ploidy + k] = haplotype index.
 * Keeping the matrix on the device and returning G numbers instead of H*R removes the D2H / gather volume. */
int phmm_genotype_likelihoods(phmm_engine* e, const double* lnl, int32_t n_haplotypes, int32_t n_reads,
                              const int32_t* genotypes, int32_t n_genotypes, int32_t ploidy, double* out, int space);

/* ---------------------------------------------------------------------------------------------------------------------
 * HaplotypeLikelihoodModel::reset (haplotype_likelihood_model.cpp:60-78): the per-haplotype penalty arrays of phmm_haplotypes
 * from the haplotype sequences, by the reference's error models — host C++ (octopus_b200/csrc/phmm_error_model.cpp), no GPU
 * needed, bit-identical to core/models/error/ (repeat_based_indel_error_model.cpp:67-83, repeat_based_snv_error_model.cpp:144-179)
 * including the exact output of the tandem-repeat finder they call (lib/tandem).
 * ------------------------------------------------------------------------------------------------------------------- */
typedef struct phmm_error_model phmm_error_model;

/* make_error_model(label) (error_model_factory.cpp:531-559): "<library>[.<sequencer>]", case-insensitive, e.g. the reference's
 * default "PCR-free.HiSeq-2500" (config/option_parser.cpp:571-573); NULL / "" = that default. Libraries PCR, PCR-free (PCRF), 10X,
 * MDA; sequencers HiSeq-2000/2500/4000, X10, NovaSeq, BGISEQ-500, PacBio, PacBioCCS (no SNV model for the last two). */
int  phmm_error_model_create(phmm_error_model** out, const char* label);
/* make_error_model(file) (:561-589): the text of a custom indel model ("MOTIF:p0,p1,..." open rows, "MOTIF+:" extension rows,
 * '#' comments; custom_repeat_based_indel_error_model.cpp:104-158) with the default SNV model. */
int  phmm_error_model_create_custom(phmm_error_model** out, const char* model_text);
void phmm_error_model_destroy(phmm_error_model* m);
const char* phmm_error_model_last_error(void);   /* thread-local message of the last failing phmm_error_model_* / phmm_reset_* call */

/* reset() for n haplotypes at once: fills the six per-base arrays (same layout as phmm_haplotypes, host memory). is_substitution:
 * optional per-base flags — bases that are substitutions in Haplotype::cigar() keep the maximum SNV prior
 * (repeat_based_snv_error_model.cpp:128-140, 166-170); NULL = none. n_threads <= 0: one per hardware thread (at most one per haplotype). */
int  phmm_reset_haplotypes(const phmm_error_model* m, int32_t n, const int64_t* off, const char* seq, const uint8_t* is_substitution,
                           char* snv_mask_fwd, int8_t* snv_prior_fwd, char* snv_mask_rev, int8_t* snv_prior_rev,
                           int8_t* gap_open, int8_t* gap_extend, int32_t n_threads);

/* tandem::extract_exact_tandem_repeats(seq, min_period, max_period) (lib/tandem/tandem.hpp:504-521): (pos, length, period) triples in
 * the library's output order. Returns the number of repeats (only the first cap are written), or a negative error code. */
int  phmm_tandem_repeats(const char* seq, int32_t n, int32_t min_period, int32_t max_period, uint32_t* out_triples, int32_t cap);

#ifdef __cplusplus
}
#endif
#endif /* PHMM_B200_H */
