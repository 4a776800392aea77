/* plink2_b200.h - C-ABI kernel face of the B200-native pairwise-genotype path.
 *
 * This is the drop-in boundary (SURVEY.md 8b, "kernel face").  It is shaped like the reference's
 * only existing GPU seam, 2.0/cuda/plink2_matrix_cuda.h:23-108: plain C, extern "C", no CUDA
 * headers leaked, opaque handles, `int` return 0 = ok / 1 = fail (the caller maps 1 to
 * kPglRetGpuFail, 2.0/include/plink2_base.h:380, as 2.0/plink2_matrix_calc.cc:9128 does),
 * idempotent cleanup, one handle per host thread / device.
 *
 * Every entry point names the reference function whose inner loop it replaces.  Data contracts
 * are the reference's own in-memory layouts so results drop into its writers unchanged:
 *
 *  - genotype block ("genovecs"): variant-major packed 2-bit genotypes exactly as PgrGet returns
 *    them (2.0/include/pgenlib_read.h:537): sample s of a variant lives in bits 2*(s%32) of
 *    64-bit word s/32 (little-endian, so also bits 2*(s%16) of 32-bit word s/16);
 *    0 = hom-REF, 1 = het, 2 = hom-ALT, 3 = missing.  Trailing entries of the last word need not
 *    be initialised (the library forces them to "missing", as SetTrailingNyps does at
 *    plink2_matrix_calc.cc:2060).
 *  - KING counts: uint32 king_counts[pair][5] in the order {IBS0, HETHET, HET2HOM1, HET1HOM2,
 *    HOMHOM} (plink2_matrix_calc.cc:864-868), pairs ordered "for row j in [row_start,row_end):
 *    for i in [0,j)" (:1545-1547); index 1 = smaller sample index, 2 = larger.
 *
 * There is no CPU fallback: every call fails (returns 1, message in pl2gpu_last_error()) when no
 * sm_100 device is usable.
 */
#ifndef PLINK2_B200_H_
#define PLINK2_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- context (replaces CudaGetDeviceCount/CudaSetDevice + CublasFmultiplier{Preinit,Init,Cleanup},
 * plink2_matrix_cuda.h:30-104) ---- */
typedef struct Pl2GpuCtx Pl2GpuCtx;

int pl2gpu_device_count(void);
/* Thread-local description of the last failure on this thread ("" if none). */
const char* pl2gpu_last_error(void);
/* Library/ABI version, bumped on any signature change. */
int pl2gpu_abi_version(void);

int pl2gpu_ctx_create(int device_idx, Pl2GpuCtx** ctx_ptr);
/* Idempotent; accepts NULL. */
int pl2gpu_ctx_destroy(Pl2GpuCtx* ctx);
/* Blocks until all work queued on the context's stream is complete. */
int pl2gpu_ctx_synchronize(Pl2GpuCtx* ctx);
/* The context's cudaStream_t as an opaque pointer (so a caller that owns device buffers, e.g. a
 * torch.distributed process, can order its own work against ours). */
void* pl2gpu_ctx_stream(Pl2GpuCtx* ctx);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
uint64_t pl2gpu_ctx_launch_count(Pl2GpuCtx* ctx);
/* Free / total device memory in bytes (pass planning, the analogue of bigstack_left()). */
int pl2gpu_ctx_mem_info(Pl2GpuCtx* ctx, uint64_t* free_bytes, uint64_t* total_bytes);
/* Page-locked host buffers for genotype blocks / results (async copies need them). */
int pl2gpu_host_alloc(uint64_t bytes, void** ptr);
int pl2gpu_host_free(void* ptr);
/* CUDA-event timing ON THE CONTEXT'S STREAM (the stream every kernel of this library is launched
 * on): record event `slot` (0..15) now; elapsed = milliseconds between two recorded slots (blocks
 * until the later one has completed). */
int pl2gpu_ctx_event_record(Pl2GpuCtx* ctx, int slot);
int pl2gpu_ctx_event_elapsed_ms(Pl2GpuCtx* ctx, int slot_from, int slot_to, float* ms);

/* ---- multi-GPU: one context (= one GPU, one rank) per process or host thread; NCCL over NVLink, loaded with
 * dlopen on first use.  The N x N outputs are row-block partitioned exactly like the reference's `--parallel`
 * pieces (ParallelBounds, 2.0/plink2_common.cc:4956-4961); the only data exchange is one all-gather of each
 * genotype column tile (pl2gpu_king_add_variants_sharded) and, for `--pca approx`, one all-reduce of the
 * N x 2k pass matrix per pass (the sum over per-thread g2_bb_part_bufs, 2.0/plink2_matrix_calc.cc:5838-5847).
 * Rank 0 creates the id, every rank passes the same bytes to pl2gpu_comm_init (collective call). ---- */
#define PL2GPU_COMM_ID_BYTES 128
int pl2gpu_comm_unique_id(uint8_t* id_out /* [PL2GPU_COMM_ID_BYTES] */);
int pl2gpu_comm_init(Pl2GpuCtx* ctx, int rank, int world, const uint8_t* id);
/* Idempotent; also called by pl2gpu_ctx_destroy. */
int pl2gpu_comm_destroy(Pl2GpuCtx* ctx);
/* In-place sum over all ranks of a device fp64 buffer, on the context's stream. */
int pl2gpu_comm_allreduce_sum_f64(Pl2GpuCtx* ctx, double* device_buf, uint64_t count);

/* ---- KING-robust pair counts: replaces the CalcKingDenseThread -> IncrKing/IncrKingHomhom hot
 * loop (plink2_matrix_calc.cc:1255-1334, :1533-1552) together with the reader-thread
 * SplitHomRef2hetUnsafeW + TransposeBitblock staging (:2055-2099).  The sparse pre-scan
 * (CalcKingSparseThread, :904-1250) is a CPU-side optimisation whose result is identical to
 * all-dense counting; here every variant goes through the dense path and the singleton vectors
 * are implicitly zero. ---- */
typedef struct Pl2KingJob Pl2KingJob;

enum {
  kPl2KingAlgoAuto = 0,
  kPl2KingAlgoPopcount = 1, /* bit-plane AND/XOR + __popc over smem tiles */
  kPl2KingAlgoTensor = 2,   /* exact int8 tcgen05 contraction over {0,+-1} indicator planes (both operands via smem) */
  kPl2KingAlgoTensorTS = 3  /* same contraction, row-side operand expanded straight into tensor memory */
};

/* Rows [row_start, row_end) of the strict lower triangle over sample_ct samples (row = larger
 * sample index), i.e. one `--parallel` piece / one TriangleLoadBalance slab.  Device accumulators
 * for those rows are allocated here; fails with "insufficient device memory" if they do not fit
 * (the caller then narrows the row range - the reference's CountTrianglePasses multipass). */
int pl2gpu_king_begin(Pl2GpuCtx* ctx, uint32_t sample_ct, uint32_t row_start, uint32_t row_end, int algo, Pl2KingJob** job_ptr);
/* Same, with the capacity of the staged genotype block chosen by the caller: every add_variants call is
 * processed in chunks of at most max_variants_per_add variants (0 = 65,536; at most 2^20; rounded up to a
 * multiple of 256).  Larger chunks amortise the per-tile accumulator read-modify-write over more variants. */
int pl2gpu_king_begin_ex(Pl2GpuCtx* ctx, uint32_t sample_ct, uint32_t row_start, uint32_t row_end, int algo, uint32_t max_variants_per_add, Pl2KingJob** job_ptr);
/* Bytes of device memory pl2gpu_king_begin_ex would need for that row range and chunk size (for pass planning,
 * the analogue of CountTrianglePasses, 2.0/plink2_matrix_calc.cc:216-255). */
uint64_t pl2gpu_king_mem_required(uint32_t sample_ct, uint32_t row_start, uint32_t row_end, uint32_t max_variants_per_add);
/* Accumulate `variant_ct` more variants.  `genovecs` is host memory unless src_is_device != 0;
 * consecutive variants are `variant_stride_bytes` apart (>= 8*ceil(sample_ct/32), multiple of 8).
 * src_is_device: 0 = host memory (the call returns once the buffer has been consumed; the kernels keep
 * running), 1 = device memory written by work the caller ordered on the context's stream, 2 = device memory
 * that is already complete (lets the copy of batch k+1 overlap the tensor kernel of batch k).  A device
 * source must stay unmodified until work queued on the context's stream after this call has started. */
int pl2gpu_king_add_variants(Pl2KingJob* job, const void* genovecs, uint64_t variant_stride_bytes, uint32_t variant_ct, int src_is_device);
/* Multi-GPU form (context with a communicator; collective call): every rank passes ITS `slice_variant_ct`
 * variants (same count on every rank - the last slice of a file is topped up by the caller with all-missing
 * rows, which count nothing); one in-place NCCL all-gather on the prep stream assembles the
 * world * slice_variant_ct-variant column tile on every GPU, overlapped with the previous batch's tensor
 * kernel.  Rank r's variants are rows [r * slice, (r + 1) * slice) of the batch. */
int pl2gpu_king_add_variants_sharded(Pl2KingJob* job, const void* slice, uint64_t variant_stride_bytes, uint32_t slice_variant_ct, int src_is_device);
/* Copy out uint32 counts[pair][5] for rows [out_row_start, out_row_end) (a sub-range of the job's
 * rows) in the reference's pair order.  dst is host memory unless dst_is_device != 0. */
int pl2gpu_king_get_counts(Pl2KingJob* job, uint32_t out_row_start, uint32_t out_row_end, uint32_t* dst, int dst_is_device);
/* Same pairs, KING-robust kinship as fp64 (ComputeKinship, plink2_matrix_calc.cc:1566-1573, with
 * zero singleton terms): 0.5 - (4*IBS0 + HET1HOM2 + HET2HOM1) / (4*(HETHET + min(HET1HOM2, HET2HOM1))). */
int pl2gpu_king_get_kinship(Pl2KingJob* job, uint32_t out_row_start, uint32_t out_row_end, double* dst, int dst_is_device);
/* `--king-table-filter` evaluated on the device: the pairs of rows [r0,r1) whose kinship is NOT below
 * min_kinship (the reference's test, 2.0/plink2_matrix_calc.cc:2296-2300), sorted in table order
 * (row j ascending, then i).  Host outputs: pairs[k][2] = {j (larger index), i}, counts[k][5], kinship[k].
 * *n_found = number of qualifying pairs; when it exceeds max_out the outputs are incomplete and the
 * call should be repeated with larger buffers. */
int pl2gpu_king_get_filtered(Pl2KingJob* job, uint32_t r0, uint32_t r1, double min_kinship, uint64_t max_out, uint32_t* pairs_out, uint32_t* counts_out, double* kinship_out, uint64_t* n_found);
uint64_t pl2gpu_king_variants_added(Pl2KingJob* job);
/* Device time of the most recent pair-count tensor kernel launch (CUDA events recorded around that launch on
 * the context's stream; blocks until it has finished).  bench.py's roofline uses it. */
int pl2gpu_king_last_kernel_ms(Pl2KingJob* job, float* ms);
/* Idempotent; accepts NULL. */
int pl2gpu_king_end(Pl2KingJob* job);

/* ---- KING counts for an explicit pair list: replaces IncrKingSubset / IncrKingSubsetHomhom
 * (2.0/plink2_matrix_calc.cc:2495-2741) driven by CalcKingTableSubset (:3224), i.e.
 * `--make-king-table --king-table-subset`.  pairs[2 p], pairs[2 p + 1] = sample indices of pair p
 * (host memory, copied at begin); counts come back as uint32 [pair][5] in the same
 * {IBS0, HETHET, HET2HOM1, HET1HOM2, HOMHOM} order, where - as in the reference's subset path - "1" is
 * the FIRST sample of the listed pair and "2" the second. ---- */
typedef struct Pl2KingPairJob Pl2KingPairJob;
int pl2gpu_king_pairs_begin(Pl2GpuCtx* ctx, uint32_t sample_ct, const uint32_t* pairs_host, uint64_t pair_ct, Pl2KingPairJob** job_ptr);
int pl2gpu_king_pairs_add_variants(Pl2KingPairJob* job, const void* genovecs, uint64_t variant_stride_bytes, uint32_t variant_ct, int src_is_device);
int pl2gpu_king_pairs_get_counts(Pl2KingPairJob* job, uint64_t pair_start, uint64_t pair_end, uint32_t* dst, int dst_is_device);
int pl2gpu_king_pairs_end(Pl2KingPairJob* job);

/* ---- GRM: replaces ExpandCenteredVarmaj + the CalcGrmThread/CalcGrmPartThread dsyrk/dgemm
 * accumulation (2.0/plink2_matrix_calc.cc:3839-3886, :4285-4327) and the CalcMissingMatrix pass
 * (:4404-4553) for rows [row_start,row_end) of the lower triangle (diagonal included), one
 * TriangleFill2 slab / `--parallel` piece.  Exact int8 tcgen05 accumulation of fixed-point
 * (32-bit) per-variant genotype tables; see DESIGN.md for the error bound. ---- */
typedef struct Pl2GrmJob Pl2GrmJob;
enum {
  kPl2GrmMeanimpute = 1, /* `meanimpute` modifier: divide by the variant count, not per-pair obs counts */
  kPl2GrmCov = 2         /* `cov` modifier: no variance standardisation (inv_stdev = 1) */
};
int pl2gpu_grm_begin(Pl2GpuCtx* ctx, uint32_t sample_ct, uint32_t row_start, uint32_t row_end, int flags, Pl2GrmJob** job_ptr);
/* ref_freqs: host double[variant_ct] REF allele frequencies (the caller's allele_freqs); NULL =
 * compute them from this block's genotype counts as ComputeAlleleFreqs does (all samples founders);
 * a NaN entry means the same for that one variant (partial --read-freq files).  The same convention
 * holds for pl2gpu_pca_add_variants and pl2_indep_pairwise[_ex].
 * Returns 2 (kPglRetDegenerateData at the call site) when a zero-variance frequency meets a
 * non-monomorphic variant, like ExpandCenteredVarmaj :3844-3868. */
int pl2gpu_grm_add_variants(Pl2GrmJob* job, const void* genovecs, uint64_t variant_stride_bytes, uint32_t variant_ct, int src_is_device, const double* ref_freqs);
/* Multi-GPU form (context with a communicator; collective call), as pl2gpu_king_add_variants_sharded: every rank
 * passes its slice_variant_ct rows, the library all-gathers the world * slice_variant_ct-row column tile; the
 * first batch_variant_ct rows of the gathered tile are the batch's variants (the rest is filler and ignored).
 * ref_freqs: host double[batch_variant_ct] for the WHOLE batch (same on every rank) or NULL. */
int pl2gpu_grm_add_variants_sharded(Pl2GrmJob* job, const void* slice, uint64_t variant_stride_bytes, uint32_t slice_variant_ct, uint32_t batch_variant_ct, int src_is_device, const double* ref_freqs);
/* Normalised relationship values (CalcGrm :4769-4788) for rows [r0,r1) in the reference's in-memory
 * layout dst_grm[(j - r0) * row_stride + i], i <= j (entries i > j are left untouched / zero);
 * dst_obs (optional) receives the per-pair observation counts as float (.grm.N.bin payload). */
int pl2gpu_grm_get_rows(Pl2GrmJob* job, uint32_t r0, uint32_t r1, double* dst_grm, float* dst_obs, uint64_t row_stride, int dst_is_device);
uint64_t pl2gpu_grm_variants_added(Pl2GrmJob* job);
/* Exact --pca (CalcPca non-approx branch, plink2_matrix_calc.cc:5942-6040 -> ExtractEigvecs/dsyevr,
 * plink2_matrix.cc:1089): top pc_ct eigenpairs of the finished GRM (job must cover all rows).
 * eigvals_host[pc_ct] descending; eigvecs_host[pc][sample], unit norm, sign arbitrary. */
int pl2gpu_grm_eigen_topk(Pl2GrmJob* job, uint32_t pc_ct, double* eigvals_host, double* eigvecs_host);
int pl2gpu_grm_end(Pl2GrmJob* job);

/* ---- `--pca approx` (CalcPca approx branch, 2.0/plink2_matrix_calc.cc:5697-5941: CalcPcaXtxaThread
 * :5210, CalcPcaXaThread :5243, CalcPcaXtbThread :5272, SvdRectFused :5860/:5918).  The whole 2-bit
 * genotype matrix stays resident in HBM; Y (standardised, missing -> 0) is never materialised.
 * g1_host: the N x 2k Gaussian start matrix, row-major [sample][2k] (FillGaussianDArr order).
 * Returns eigvals[pc_ct] = sigma^2 / M and eigvecs[pc][sample].  Return code 2 = kPglRetDegenerateData. ---- */
typedef struct Pl2PcaJob Pl2PcaJob;
int pl2gpu_pca_begin(Pl2GpuCtx* ctx, uint32_t sample_ct, uint32_t variant_ct_total, uint32_t pc_ct, Pl2PcaJob** job_ptr);
int pl2gpu_pca_add_variants(Pl2PcaJob* job, const void* genovecs, uint64_t variant_stride_bytes, uint32_t variant_ct, int src_is_device, const double* ref_freqs);
int pl2gpu_pca_run(Pl2PcaJob* job, const double* g1_host, double* eigvals_host, double* eigvecs_host);
/* Multi-GPU form (contexts joined by pl2gpu_comm_init; collective call, one host thread per rank): every rank's job
 * holds ONE shard of the variants (any split; begin / add_variants as above with the shard's own variant count),
 * total_variant_ct = the sum over ranks.  H_t = Y G_t stays on the rank that owns the variants; G' = Y^T H is completed by
 * one fp64 all-reduce of the N x 2k matrix per pass (SURVEY 8e), likewise the Gram-Schmidt coefficients and B = Y^T Q;
 * each M x 2k block of the basis construction is all-gathered for the (replicated) Jacobi SVD.  Every rank returns
 * the same eigenvalues / eigenvectors. */
int pl2gpu_pca_begin_shard(Pl2GpuCtx* ctx, uint32_t sample_ct, uint32_t shard_variant_ct, uint32_t pc_ct, Pl2PcaJob** job_ptr);
int pl2gpu_pca_run_sharded(Pl2PcaJob* job, const double* g1_host, uint64_t total_variant_ct, double* eigvals_host, double* eigvecs_host);
/* `--variant-score` (VscoreReport, 2.0/plink2_matrix_calc.cc:9274) on the resident matrix of a Pl2PcaJob (begin +
 * add_variants as above; pc_ct is irrelevant): out_host[variant][cols] = sum over samples of weights_host[sample][cols]
 * x ALT dosage, a missing call replaced by 2 x the variant's ALT frequency (the ref_freqs given to add_variants, else
 * the block's own).  Samples that are not scored get weight 0.  One H = Y W pass of the int8 tensor tile path plus an
 * un-standardising epilogue; any number of score columns (48 per launch). */
int pl2gpu_pca_vscore(Pl2PcaJob* job, const double* weights_host, uint32_t cols, double* out_host);
int pl2gpu_pca_end(Pl2PcaJob* job);

/* ---- per-variant genotype counts {hom-REF, het, hom-ALT, missing}: the hard-call part of the
 * LoadAlleleAndGenoCounts pre-pass (2.0/plink2.cc:2280; GenoarrCountFreqsUnsafe,
 * 2.0/include/pgenlib_misc.cc:702) that feeds ComputeAlleleFreqs (2.0/plink2_filter.cc:2113).
 * counts_host: uint32 [variant_ct][4] (host memory). ---- */
int pl2gpu_geno_counts(Pl2GpuCtx* ctx, const void* genovecs, uint64_t variant_stride_bytes, uint32_t sample_ct, uint32_t variant_ct, int src_is_device, uint32_t* counts_host);

/* ---- --indep-pairwise pair decisions: replaces ComputeIndepPairwiseR2Components (DotprodWords /
 * SumSsqWords / SumSsqNmWords, 2.0/plink2_ld.cc:699-723, :235, :317, :578) and the r^2 test
 * (:1085-1090) for every pair that can share a window.  flags_host[v * band + (d - 1)], 1 <= d <= band,
 * is 1 iff for second = v, first = v - d:  cov12^2 > prune_ld_thresh * var1 * var2  (exact int64
 * sextuple -> fp64, unfused multiplies).  genovecs: founders only, PgrGet layout.  Besides the LD prune, the same
 * call is the screening pass of `--r2-unphased` tables (threshold set a hair below --ld-window-r2; the few flagged
 * pairs are then finished on the host with ComputeR2's arithmetic, 2.0/plink2_ld.cc:6654-6682). ---- */
int pl2gpu_ld_band_flags(Pl2GpuCtx* ctx, const void* genovecs, uint64_t variant_stride_bytes, uint32_t founder_ct, uint32_t variant_ct, int src_is_device, uint32_t band, double prune_ld_thresh, uint8_t* flags_host);

/* ---- function face of LdPrune -> IndepPairwise (2.0/plink2_ld.h:160, 2.0/plink2_ld.cc:2530, :1116)
 * on an in-memory founder genotype block: variants in file order with chromosome codes (0 =
 * unplaced, never examined), bp positions (needed iff window_is_bp), window/step/r^2 as parsed from
 * `--indep-pairwise`, optional REF allele frequencies (NULL = compute from the block, as
 * ComputeAlleleFreqs does) and optional --indep-preferred flags.  removed_out[v] = 0 kept
 * (.prune.in), 1 removed (.prune.out), 2 unplaced.  The GPU evaluates the pair decisions; the greedy
 * window walk (IndepPairwiseThread, :862-1109) runs on the calling host thread. ---- */
int pl2_indep_pairwise(Pl2GpuCtx* ctx, const void* genovecs, uint64_t variant_stride_bytes, uint32_t founder_ct, uint32_t variant_ct, const uint32_t* chr_codes, const uint32_t* variant_bps, uint32_t window_size, uint32_t window_incr, double r2_thresh, int window_is_bp, const double* ref_freqs, const uint8_t* preferred, int src_is_device, uint8_t* removed_out);

/* Extended form: founder_sex[founder_ct] (0 unknown, 1 male, 2 female; NULL = all unknown) selects the reference's
 * sex-chromosome handling (IndepPairwise loader, 2.0/plink2_ld.cc:1356-1389; sums :982-998): chrX (code 23) = males
 * with hets -> missing at weight 1 plus nonmales at weight 2, chrY (24) = nonfemale founders with hets -> missing,
 * MT (26) = all founders with hets -> missing; allele frequencies follow LoadAlleleAndGenoCountsThread's per-class
 * counting (2.0/plink2_data.cc:2420-2690).  flags: kPl2LdPlink1Order = `--indep-order 1` (:931-1037). */
enum { kPl2LdPlink1Order = 1 };
int pl2_indep_pairwise_ex(Pl2GpuCtx* ctx, const void* genovecs, uint64_t variant_stride_bytes, uint32_t founder_ct, uint32_t variant_ct, const uint32_t* chr_codes, const uint32_t* variant_bps, uint32_t window_size, uint32_t window_incr, double r2_thresh, int window_is_bp, const double* ref_freqs, const uint8_t* preferred, int src_is_device, const uint8_t* founder_sex, uint32_t flags, uint8_t* removed_out);
/* Host half of the function face on its own (no device work): IndepPairwiseThread's greedy window walk
 * (2.0/plink2_ld.cc:862-1109, window bookkeeping :605-689, subcontigs :2165-2268) over precomputed pair
 * decisions pair_flags[v * band + d - 1] (second = v, first = v - d; band >= widest window - 1), load-time
 * monomorphic marks (:902) and major-allele frequencies (minus 1 for --indep-preferred variants, :916-918). */
int pl2_ld_prune_walk(uint32_t variant_ct, const uint32_t* chr_codes, const uint32_t* variant_bps, uint32_t window_size, uint32_t window_incr, int window_is_bp, const double* maj_freq, const uint8_t* mono, const uint8_t* pair_flags, uint32_t band, uint32_t flags, uint8_t* removed_out);

/* ---- `--score`: replaces the per-variant dosage expansion + dgemm / difflist updates of CalcScoreThread
 * (2.0/plink2_matrix_calc.cc:6467-6890) under ScoreReport (:6892) for diploid hard calls.  Entries (one per scored
 * (variant, allele) line, in any order) are streamed as PgrGet rows together with, per entry, weights4[e][code] =
 * the contribution of genotype code 0/1/2/3 (code 3 = missing: coefficient x 2 x named-allele frequency, or 0 with
 * 'no-mean-imputation', :6605-6607) and named_dosages[e] = the named-allele dosages of codes 0, 1, 2 packed two
 * bits each (bits 0-1, 2-3, 4-5): 0x24 when the ALT allele is named, 0x06 when REF is ('dominant': 0x14 / 0x05,
 * 'recessive': 0x10 / 0x01).  pl2gpu_score_get returns per sample the weighted sum, the named-allele dosage
 * sum over nonmissing calls (NAMED_ALLELE_DOSAGE_SUM) and the number of missing calls (ALLELE_CT = 2 x (entries -
 * missing), :8581).  Partial sums are combined in a fixed order: results are bit-reproducible. ---- */
typedef struct Pl2ScoreJob Pl2ScoreJob;
int pl2gpu_score_begin(Pl2GpuCtx* ctx, uint32_t sample_ct, Pl2ScoreJob** job_ptr);
int pl2gpu_score_add_variants(Pl2ScoreJob* job, const void* genovecs, uint64_t variant_stride_bytes, uint32_t variant_ct, int src_is_device, const double* weights4, const uint8_t* named_dosages);
int pl2gpu_score_get(Pl2ScoreJob* job, double* score_sums, uint64_t* named_dosage_sums, uint32_t* missing_cts);
/* Idempotent; accepts NULL. */
int pl2gpu_score_end(Pl2ScoreJob* job);

/* ---- measured int8 tensor peak: every SM issues back-to-back tcgen05.mma kind::i8 (M = 128, N = n_cols,
 * K = 32; form 0 = both operands in shared memory, 1 = A operand in tensor memory as the KING/GRM kernels use
 * it) for at least min_seconds; *tops_out = 2*128*n_cols*32 ops x UMMAs / elapsed (CUDA events), in TOP/s.
 * This is the roofline denominator bench.py reports against. ---- */
int pl2gpu_int8_peak(Pl2GpuCtx* ctx, uint32_t n_cols, int form, double min_seconds, double* tops_out, double* seconds_out);

/* ---- measured block-scaled FP4 tensor peak: as pl2gpu_int8_peak's form 1, with tcgen05.mma kind::mxf4
 * (E2M1 operands, UE8M0 scales, M = 128, N = n_cols, K = 64, A operand in tensor memory as king_ts_kernel uses it);
 * *tops_out = 2*128*n_cols*64 ops x UMMAs / elapsed, in TOP/s. ---- */
int pl2gpu_mxf4_peak(Pl2GpuCtx* ctx, uint32_t n_cols, double min_seconds, double* tops_out, double* seconds_out);

/* ---- self-test of the tcgen05 operand path (descriptor/layout probe); returns 0 iff int8 UMMAs (both
 * operands in shared memory, and A in tensor memory) and kind::mxf4 UMMAs in king_ts_kernel's operand layout
 * reproduce a scalar reference, and the kind::mxf4 F32 accumulator adds +-1 exactly past 2^20. ---- */
int pl2gpu_selftest_umma(Pl2GpuCtx* ctx, int verbose);
/* Debug probe used by tests to pin the operand layout: runs `k_steps` int8 UMMAs (M = 128) over the
 * given shared-memory images / descriptor fields and returns D as int32 [128][n] (host memory). */
int pl2gpu_debug_umma(Pl2GpuCtx* ctx, const uint8_t* a_img, uint32_t a_bytes, const uint8_t* b_img, uint32_t b_bytes, uint32_t a_lbo, uint32_t a_sbo, uint32_t b_lbo, uint32_t b_sbo, uint32_t a_step_bytes, uint32_t b_step_bytes, uint32_t k_steps, uint32_t idesc, uint32_t n, int32_t* d_out_host);

#ifdef __cplusplus
}
#endif

#endif  /* PLINK2_B200_H_ */
