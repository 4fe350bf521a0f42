/*
 * dnaf_b200.h -- C ABI of the B200-native dna-factory population-generation hot path.
 *
 * The reference (ochrzan/dna-factory) has no FFI: its seam for this path is the Python method
 *     PopulationFactory.write_vcf_snps(self, fam_data, snps, file)          pop_factory.py:417-469
 * which forks workers running
 *     PopulationFactory.queue_vcf_snps(self, fam_data, work_q, result_p)    pop_factory.py:471-513
 * and feeds their rows, in SNP order, to Bio.bgzf.BgzfWriter.write()       pop_factory.py:449
 * (opened at pop_factory.py:403, closed by the `with` at :403-413).
 * This header is what a ctypes binding of that seam needs: plain pointers and sizes, no Python
 * objects, no torch types.  INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - every function returns 0 on success or a negative DNAF_E_* code; dnaf_last_error() gives text
 *   - one context per GPU, used from one host thread at a time
 *   - the caller owns every input buffer for the duration of the call only; the library copies
 *   - output buffers are host memory owned by the caller unless the name says "device"
 *   - rows are addressed by their GLOBAL index in the sorted SNP list (pop_factory.py:245); that
 *     index is also the row word of the Philox counter, so any row range can be regenerated alone
 */
#ifndef DNAF_B200_H
#define DNAF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DNAF_ABI_VERSION 5
#define DNAF_KMAX 4 /* alleles per SNP the device path handles (A,C,G,T); K=2 for SnpFactory output */

/* chromosome classes -- the only thing is_haploid() (common/snp.py:102-109) looks at */
#define DNAF_CLASS_AUTO 0 /* diploid for everybody:          "a/b\t"  4 bytes per sample            */
#define DNAF_CLASS_X 1    /* haploid for males:              2 bytes male, 4 bytes female           */
#define DNAF_CLASS_Y 2    /* haploid; females print ".":     2 bytes per sample  (pop_factory.py:481) */
#define DNAF_CLASS_MT 3   /* haploid for everybody:          2 bytes per sample                     */

#define DNAF_OK 0
#define DNAF_E_ARG (-1)    /* bad argument / call order                    */
#define DNAF_E_CUDA (-2)   /* CUDA runtime error (message has the detail)  */
#define DNAF_E_NOMEM (-3)  /* host or device allocation failed             */
#define DNAF_E_SPACE (-4)  /* caller's output buffer too small             */
#define DNAF_E_SINK (-5)   /* the sink callback returned non-zero          */
#define DNAF_E_INPUT (-6)  /* input the reference would raise on (e.g. CDF that does not reach 1.0) */

typedef struct dnaf_ctx dnaf_ctx;

/* Ordered output callback: receives consecutive pieces of the BGZF stream (whole blocks). */
typedef int (*dnaf_sink_fn)(void* user, const uint8_t* data, uint64_t n_bytes);

typedef struct dnaf_stats {
    uint64_t rows;             /* SNP rows generated                                       */
    uint64_t calls;            /* genotype calls = rows * samples                          */
    uint64_t text_bytes;       /* uncompressed VCF text bytes of those rows                */
    uint64_t bgzf_bytes;       /* compressed bytes emitted (no EOF block)                  */
    uint64_t bgzf_blocks;      /* BGZF blocks emitted                                      */
    uint32_t crc_xor;          /* xor of all block CRC32s ("checksum of checksums")        */
    uint32_t kernel_launches;  /* kernels of this library launched by the call             */
    float ms_sample;           /* CUDA-event time of the sampling kernels                  */
    float ms_format;           /* ... of the text formatter                                */
    float ms_deflate;          /* ... of the BGZF encoder (+ compaction)                   */
    float ms_fused;            /* ... of the fused sample+format+deflate kernel            */
    float ms_total;            /* first launch to last kernel end, on the library stream   */
    float ms_auto;             /* ... of the k_auto launches alone (the dominant kernel)    */
    uint32_t auto_launches;    /* k_auto launches of the call                               */
    uint64_t auto_text_bytes;  /* uncompressed text bytes those launches emitted            */
} dnaf_stats;

int dnaf_abi_version(void);
/* CUDA devices visible to the process (0 when there is none or the driver is missing): lets the host spread the
 * contiguous SNP ranges of a multi-GPU run (pop_factory.py:426 stripes over worker processes) over what exists. */
int dnaf_device_count(void);
const char* dnaf_last_error(const dnaf_ctx* ctx); /* ctx may be NULL: error of the last failed create */

/* Replaces the worker pool set-up of write_vcf_snps (pop_factory.py:419-434). */
int dnaf_create(int device_ordinal, dnaf_ctx** out);
void dnaf_destroy(dnaf_ctx* ctx);
/* Launch on a caller-provided cudaStream_t (e.g. torch's current stream) instead of the private one. */
int dnaf_set_stream(dnaf_ctx* ctx, void* cuda_stream);
/* Upper bound on the uncompressed text handled per internal pass (default 1 GiB; tests shrink it). */
int dnaf_set_chunk_bytes(dnaf_ctx* ctx, uint64_t text_bytes);
/* Philox row counter of local row r is row_base + r (default 0): lets a process that holds only a slice
 * of the sorted SNP list, e.g. one rank of a multi-GPU run, draw the rows it was given. */
int dnaf_set_row_base(dnaf_ctx* ctx, uint64_t row_base);
/* 0 = three-kernel path only (sample -> format -> deflate), 1 = fused kernel where it applies (default). */
int dnaf_set_fused(dnaf_ctx* ctx, int enable);

/*
 * fam_data (pop_factory.py:341-383): sex[i] is SampleInfo.sex (1 = male, anything else female,
 * pop_factory.py:70-71); is_control[i] is SampleInfo.is_control.  n_samples may be 0 (sites-only run).
 */
int dnaf_set_samples(dnaf_ctx* ctx, uint32_t n_samples, const uint8_t* sex, const uint8_t* is_control);

/*
 * The sorted SNP list (SNPTuples, pop_factory.py:74-133), flattened:
 *   chrom_class[r]   DNAF_CLASS_* of snp.chromosome
 *   n_alleles[r]     len(snp.tuples), 1..DNAF_KMAX
 *   thresholds[r*4+k] floor(cum_k * 2^32) saturated to 0xFFFFFFFF when cum_k >= 1.0, so that
 *                    `tuples[k][1] >= u` (pop_factory.py:94) becomes the integer test U <= threshold
 *                    for u = U * 2^-32; entries k >= n_alleles are ignored
 *   prefix_bytes / prefix_off[r..r+1]  the 9-column row lead exactly as pop_factory.py:503-507 formats it
 * The last allele of a row takes whatever its table leaves above the last cumulative probability.  Returns
 * DNAF_E_INPUT when that last value is below 0.999 (a broken table: the reference's pick_allele_index would return
 * None and "%i" would raise as soon as a roll lands there); values that merely round short of 1.0 are accepted with
 * a one-line note on stderr.
 */
int dnaf_set_snps(dnaf_ctx* ctx, uint64_t n_snps, const uint8_t* chrom_class, const uint8_t* n_alleles,
                  const uint32_t* thresholds, const uint8_t* prefix_bytes, const uint64_t* prefix_off);

/*
 * Cells where the reference takes its forced-minor branch (pop_factory.py:485,495-499): sample is a
 * case AND `snp.id in sample.deleterious_snps`.  Pairs (global row, sample index), sorted by row.
 * The host computes them with the reference's own dict-membership semantics (SURVEY R8).
 */
int dnaf_set_overrides(dnaf_ctx* ctx, uint64_t n_pairs, const uint64_t* snp_row, const uint32_t* sample_idx);

/*
 * SNP selection: SnpFactory.random_snp_tuples (pop_factory.py:160-193) as a GPU inverse-CDF sampler, followed
 * (sorted != 0) by the stable sort on (chromosome label as a STRING, position) of pop_factory.py:245.
 *   chrom_cdf[n_chrom]      cumulative CHROMOSOME_PROB as numpy.random.choice builds it (cumsum / last)
 *   chrom_max_pos[n_chrom]  CHROMOSOME_MAX_POSITION, in CHROMOSOME_LIST order (common/snp.py:36-60)
 *   chrom_rank[n_chrom]     rank of each label in string order ("1" < "10" < ... < "2" < ... < "X" < "Y")
 *   maf_cdf[n_maf]          cumulative pdf[start:]/sum of the MAF grid from the -f bin on (pop_factory.py:160-167)
 * Draw n (SNP id = n + 1) takes five uniforms from the counter-based stream (DESIGN.md 3); outputs are columns in
 * final order: order[r] = draw index of row r, chrom_idx[r] (index into CHROMOSOME_LIST), maf_bin[r] (index into
 * the grid slice), position[r], ref[r] / alt[r] (ASCII nucleotides).  Any n gives the same SNP for the same n.
 */
int dnaf_select_snps(dnaf_ctx* ctx, uint64_t n_snps, uint64_t seed, uint32_t n_chrom, const double* chrom_cdf,
                     const double* chrom_max_pos, const uint8_t* chrom_rank, uint32_t n_maf, const double* maf_cdf,
                     int sorted, uint32_t* order, uint8_t* chrom_idx, uint8_t* maf_bin, uint32_t* position,
                     uint8_t* ref, uint8_t* alt);

/*
 * load_snps_file (pop_factory.py:264-272) without a Python object per SNP: parses the inflated snps.json text
 * (one SNPTuples.__str__ record per line, pop_factory.py:118-124) into columns.  Host code, no context needed.
 * nts / cum are [cap][DNAF_KMAX] (unused entries 0 / 2.0; the order of "tuples" is kept); chrom_labels receives up to
 * max_labels labels of <= 7 characters, 8 bytes each, in order of first appearance.  Returns the number of
 * records, or -(line number) at the first record the column form cannot hold (the caller falls back to json.loads).
 */
int64_t dnaf_parse_snps_jsonl(const char* text, uint64_t n_bytes, uint64_t cap, int64_t* ids, int32_t* chrom_idx,
                              int64_t* position, uint8_t* n_alleles, uint8_t* nts, double* cum, char* chrom_labels,
                              uint32_t max_labels, uint32_t* n_labels);

/*
 * Host-side formatters for column-form SNP tables (no context needed; `labels` = 8 bytes per chromosome label).
 * dnaf_format_prefixes: the row leads "%s\t%i\trs%s\t%s\t%s\t40\tPASS\t.\tGT\t" of pop_factory.py:503-507 (ALT as
 *   SNPTuples.alt_alleles, pop_factory.py:111-116) into `out` (caller sizes it: <= 64 + 8 bytes per row), offsets in
 *   off[n+1]; returns the bytes written.  Ids and positions must be non-negative.
 * dnaf_format_snps_jsonl: the snps.json lines of SNPTuples.__str__ (pop_factory.py:118-124); floats come from the
 *   caller's table of Python reprs (repr_idx[r*4+j] -> reprs + repr_off[...], NUL-terminated).  Returns bytes written.
 */
uint64_t dnaf_format_prefixes(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* position,
                              const int64_t* ids, const uint8_t* n_alleles, const uint8_t* nts, char* out, uint64_t* off);
uint64_t dnaf_format_snps_jsonl(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* position,
                                const int64_t* ids, const uint8_t* n_alleles, const uint8_t* nts, const uint32_t* repr_idx,
                                const char* reprs, const uint32_t* repr_off, char* out);

/* Sizes of rows [row_begin,row_end): exact text bytes and an upper bound on the BGZF bytes. */
int dnaf_plan(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t* text_bytes, uint64_t* bgzf_bound);
/* out[i] = text offset of row row_begin+i relative to row row_begin, i = 0 .. row_end-row_begin (one past the
 * last row included): the row lengths queue_vcf_snps would produce (pop_factory.py:503-508), for indexing. */
int dnaf_row_offsets(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t* out);

/*
 * The hot path: rows [row_begin,row_end) -> genotype draws -> VCF text -> BGZF blocks.
 * Emits whole BGZF blocks that decompress to exactly the text of those rows (first block starts
 * and last block ends on a row boundary; no header, no EOF block -- the caller writes those).
 * There is ONE uniform stream, the counter-based Philox stream of DESIGN.md 3: what a "replay" of the reference is fed
 * and what a production ("native") run draws are the same function of (seed, global row, allele slot); ABI 4's
 * rng_mode argument selected nothing and is gone.
 * level: the -z value the reference hands to BgzfWriter (pop_factory.py:403; default 6, :656-658).  1..3 = the
 * byte-4-back parse (k_auto), 4..9 = LZ77 tiers of growing search depth on autosome rows (k_lz: hash chains of
 * 1 / 4 / 16 / 16+lazy / 32+lazy / 128+lazy candidates).  The decompressed text does not depend on it.
 */
int dnaf_generate(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level,
                  uint8_t* out, uint64_t out_cap, dnaf_stats* stats);
int dnaf_generate_stream(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level,
                         dnaf_sink_fn sink, void* user, dnaf_stats* stats);
/* Same work, every piece written to an open file descriptor (the ordered `file.write(line)` loop of
 * pop_factory.py:438-469 without a trip through the interpreter); the caller flushes its own buffers first. */
int dnaf_generate_fd(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level,
                     int fd, dnaf_stats* stats);
/* Same, written with pwrite() at file_offset (the descriptor's own position is neither used nor moved): ranks of a
 * multi-GPU run that know their streams' sizes (a dnaf_generate_device pass gives bgzf_bytes) write one shared file
 * side by side, in SNP order, without spooling (pop_factory.py:426 stripes SNPs over workers the same way). */
int dnaf_generate_fd_at(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level, int fd,
                        uint64_t file_offset, dnaf_stats* stats);
/* Same work, output left in (and then discarded from) device memory: kernel-only timing. */
int dnaf_generate_device(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, int level,
                         dnaf_stats* stats);

/*
 * PLINK 1 binary genotypes (.bed) of rows [row_begin,row_end): the same draws, forced minors and ploidy rules as the
 * VCF rows of the same seed (pop_factory.py:481-499), so population.bed and population.vcf.gz describe one population.
 * Payload only: ceil(n_samples/4) bytes per row, SNP-major, no magic bytes (the caller writes 6C 1B 01 first, like it
 * writes the VCF header).  Sample i sits in byte i/4 at bits 2(i%4), 2(i%4)+1; padding bits are 0.  Values count ALT
 * copies with .bim A1 = ALT, A2 = REF: 2 copies -> 0, 1 -> 2, 0 -> 3, missing ('.', females on Y) -> 1; haploid cells
 * are written homozygous.  Rows with more than 2 alleles cannot be written: DNAF_E_INPUT before any GPU work, naming
 * the row.  stats: rows, calls, kernel_launches, ms_sample (the .bed kernel), ms_total; the other fields are 0.
 */
int dnaf_generate_bed(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint8_t* out, uint64_t out_cap,
                      dnaf_stats* stats);
/* Same bytes written with pwrite() at file_offset (3 + first row * ceil(n_samples/4) in population.bed). */
int dnaf_generate_bed_fd_at(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, int fd,
                            uint64_t file_offset, dnaf_stats* stats);
/* Same work, output left in device memory: kernel-only timing. */
int dnaf_generate_bed_device(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, dnaf_stats* stats);

/*
 * Case/control allele counts of rows [row_begin,row_end), the input of the 1-df allelic association test (plink
 * --assoc): the same draws, forced minors and ploidy rules as the VCF and .bed rows of the same seed.  counts is
 * [rows][4]: ALT alleles in cases, alleles observed in cases, ALT alleles in controls, alleles observed in controls
 * (cases: is_control[i] == 0 in dnaf_set_samples).  Every allele the VCF text prints counts once: autosome rows count
 * both slots of every sample; X rows slot 0 of males and both slots of females; Y rows slot 0 of males and nothing of
 * females ('.'); MT rows slot 0 of every sample.  A forced minor counts as ALT on every counted slot of its cell.  Rows
 * with more than 2 alleles: DNAF_E_INPUT before any GPU work, naming the row; K = 1 rows count ALT only where a minor
 * is forced.  stats: rows, calls, kernel_launches, ms_sample (the counting kernel), ms_total; the other fields are 0.
 */
int dnaf_allele_counts(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t* counts,
                       dnaf_stats* stats);
/* Same work, counts left in device memory: kernel-only timing. */
int dnaf_allele_counts_device(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, dnaf_stats* stats);
/*
 * The .assoc body lines of n rows from their counts (host code, no context, no GPU; `labels` = 8 bytes per chromosome
 * label, nts = [n][DNAF_KMAX]).  With a = ALT and b = REF alleles in cases, c / d the same in controls:
 *   F_A = a/(a+b), F_U = c/(c+d), CHISQ = n(ad-bc)^2 / ((a+b)(c+d)(a+c)(b+d)) (no continuity correction),
 *   P = erfc(sqrt(CHISQ/2)), OR = ad/(bc); "NA" where a denominator is 0; values printed with "%.4g" in double.
 * Columns CHR SNP BP A1 F_A F_U A2 CHISQ P OR, right-aligned, one space apart; CHR is the label with X, Y, MT written
 * 23, 24, 26; SNP is rs<id>; A1 = ALT ('0' for one-allele rows) and A2 = REF, as in the .bim.  `out` holds at least
 * 192 bytes per row.  Returns the bytes written.
 */
uint64_t dnaf_format_assoc(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                           const int64_t* position, const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts,
                           char* out);

/*
 * Case/control genotype counts of rows [row_begin,row_end), the input of the genotypic tests (plink --model) and of
 * the Hardy-Weinberg exact tests (plink --hardy): the same draws, forced minors and ploidy rules as the VCF and .bed
 * rows of the same seed.  counts is [rows][10]: for the cases (is_control[i] == 0 in dnaf_set_samples) dip (diploid
 * cells), het (diploid 0/1), hom (diploid 1/1, ALT/ALT), hap (haploid cells printed), hap_alt (haploid cells printed
 * as ALT); then the same five for the controls.  Diploid cells: every sample on autosome rows, females on X rows;
 * haploid cells: males on X and Y rows, every sample on MT rows; female Y cells ('.') count nothing.  A forced minor
 * makes its cell 1/1 (ALT on a haploid cell).  So 2 hom + het + hap_alt and 2 dip + hap are the ALT and observed
 * allele counts of dnaf_allele_counts.  hwe_p (NULL: not computed) is [rows][3]: the two-sided Hardy-Weinberg exact P
 * (dnaf_hwe_exact) of the diploid genotypes of ALL samples, the cases (AFF) and the controls (UNAFF); NaN where the
 * group has no diploid cell (Y and MT rows, empty groups).  Rows with more than 2 alleles: DNAF_E_INPUT before any GPU
 * work, naming the row.  stats: rows, calls, kernel_launches, ms_sample (the counting and exact-test kernels),
 * ms_total; the other fields are 0.
 */
int dnaf_genotype_counts(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t* counts,
                         double* hwe_p, dnaf_stats* stats);
/* Same work, counts (and, with with_hwe != 0, the exact tests) left in device memory: kernel-only timing. */
int dnaf_genotype_counts_device(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, int with_hwe,
                                dnaf_stats* stats);
/*
 * Two-sided Hardy-Weinberg exact P of n genotype triples geno[i] = (n11, n12, n22) (ALT/ALT, het, REF/REF), computed
 * on the device by the kernel dnaf_genotype_counts uses: Wigginton, Cutler & Abecasis (2005), the SNPHWE definition
 * of plink --hardy.  P is the sum of the probabilities of every het count whose probability is <= (1 + 1e-7) times
 * that of the observed one (the relative tolerance makes ties independent of rounding), over the sum of all of them,
 * in double precision; 0 where P < 1e-290, NaN where n11 + n12 + n22 = 0.  Synchronous.
 */
int dnaf_hwe_exact(dnaf_ctx* ctx, uint64_t n, const uint32_t* geno, double* p);
/*
 * The counts, Hardy-Weinberg P and Fisher exact tests of rows [row_begin,row_end) in one call: counts and hwe_p as in
 * dnaf_genotype_counts; fisher_log10p (NULL: not computed) is [rows][4], log10 of the two-sided Fisher exact P
 * (dnaf_fisher_exact) of GENO (the diploid 2x3 table n11 / n12 / n22 of cases and controls), ALLELIC (ALT / REF
 * alleles, haploid cells included, as in .assoc), DOM (n11 + n12 / n22) and REC (n11 / n12 + n22), each computed on
 * the device from the pass's counts.  Y and MT rows have no diploid cell, so only their ALLELIC test is defined (the
 * others are NaN).  A NULL hwe_p or fisher_log10p is not computed.  dnaf_genotype_counts is this call with
 * fisher_log10p = NULL.  Rows with more than 2 alleles: DNAF_E_INPUT before any GPU work, naming the row.
 */
int dnaf_genotype_tests(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t* counts,
                        double* hwe_p, double* fisher_log10p, dnaf_stats* stats);
/* Same work, results left in device memory (the exact tests only where with_hwe / with_fisher != 0). */
int dnaf_genotype_tests_device(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, int with_hwe,
                               int with_fisher, dnaf_stats* stats);
/*
 * log10 of the two-sided Fisher exact P of n case/control tables, tables[i] = (x1, x2, x3, y1, y2, y3) (case row, then
 * control row), computed on the device by the kernel dnaf_genotype_tests uses.  With both margins fixed a table has
 * probability prod_j C(x_j + y_j, x_j) / C(N, R); P is the sum of the probabilities of every table whose probability
 * is <= (1 + 1e-7) times the observed one's (the tie rule of dnaf_hwe_exact).  A table with one empty column is the 2x2
 * test over the other two.  Double precision, with the scale of P kept in a separate exponent, so log10 P stays exact
 * far below the double range; NaN where a row margin is 0 or fewer than two columns are non-empty.  Synchronous.
 */
int dnaf_fisher_exact(dnaf_ctx* ctx, uint64_t n, const uint32_t* tables, double* log10p);
/*
 * The .assoc.fisher body lines of n rows from their genotype counts and Fisher log10 P (dnaf_genotype_tests; labels
 * and nts as in dnaf_format_assoc): columns CHR SNP BP A1 F_A F_U A2 P OR (PLINK 1.9's plink.assoc.fisher), F_A, F_U
 * and OR from the allele counts as in .assoc, P the Fisher ALLELIC P printed "%.4g" (0 where 10^log10P underflows, NA
 * for NaN).  `out` holds at least 192 bytes per row.  Returns the bytes written.
 */
uint64_t dnaf_format_assoc_fisher(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                                  const int64_t* position, const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts,
                                  const double* log10p, char* out);
/*
 * The Fisher .model body lines (plink --model fisher): five lines a row, GENO, TREND, ALLELIC, DOM, REC, with columns
 * CHR SNP A1 A2 TEST AFF UNAFF P; AFF and UNAFF as in dnaf_format_model.  TREND prints its asymptotic chi-square P; the
 * others print the Fisher P of log10p, with no cell rule, as in dnaf_format_assoc_fisher.  `out` holds at least 960
 * bytes per row.  Returns the bytes written.
 */
uint64_t dnaf_format_model_fisher(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids,
                                  const uint8_t* nts, const uint8_t* n_alleles, const uint32_t* counts, const double* log10p,
                                  char* out);
/*
 * The .model body lines of n rows from their genotype counts (host code, no context, no GPU; labels and nts as in
 * dnaf_format_assoc): five lines a row, GENO, TREND, ALLELIC, DOM, REC, with columns CHR SNP A1 A2 TEST AFF UNAFF
 * CHISQ DF P.  With n11 / n12 / n22 the diploid ALT/ALT, het and REF/REF counts of a group, AFF and UNAFF are
 * n11/n12/n22 (GENO, TREND), ALT/REF alleles with haploid cells (ALLELIC), n11+n12/n22 (DOM), n11/n12+n22 (REC).
 * ALLELIC is the .assoc statistic; TREND the Cochran-Armitage trend test on diploid cells; GENO the 2x3 Pearson
 * test (2 df), DOM and REC 2x2 Pearson tests (1 df); no continuity correction, P the chi-square survival in double.
 * GENO, DOM and REC are NA when any of the six genotype cells is below 5 (PLINK's --cell 5); any zero denominator is
 * NA; an NA test prints NA for CHISQ, DF and P.  `out` holds at least 960 bytes per row.  Returns the bytes written.
 */
uint64_t dnaf_format_model(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids, const uint8_t* nts,
                           const uint8_t* n_alleles, const uint32_t* counts, char* out);
/*
 * The .hwe body lines of n rows from their genotype counts and hwe_p (dnaf_genotype_counts): three lines a row, ALL,
 * AFF, UNAFF, with columns CHR SNP TEST A1 A2 GENO O(HET) E(HET) P; GENO is n11/n12/n22 of the diploid cells (females
 * only on X rows, 0/0/0 on Y and MT rows), O(HET) = n12 / n and E(HET) = 2 f (1 - f) with f = (2 n11 + n12) / 2n;
 * NA where n = 0.  `out` holds at least 576 bytes per row.  Returns the bytes written.
 */
uint64_t dnaf_format_hardy(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids, const uint8_t* nts,
                           const uint8_t* n_alleles, const uint32_t* counts, const double* hwe_p, char* out);

/*
 * Case/control permutations of the samples of dnaf_set_samples (max(T) permutation tests).  Permutation p is a
 * uniformly random subset of exactly ncase of the N samples (ncase = samples with is_control == 0), by selection
 * sampling: for i = 0..N-1, with `need` starting at ncase, sample i is a case iff
 *   (uint64)U(p,i) * (N - i) < (uint64)need << 32   (then need -= 1),
 *   U(p,i) = philox4x32_10(ctr = (i >> 2, p, 0x4D505200, 0xFFFFFFFF), key = (seed_lo, seed_hi))[i & 3].
 * This call writes permutations first_perm .. first_perm + n_perm - 1 (indices below 2^32): masks is
 * [n_perm][ceil(N/32)], bit i & 31 of word i >> 5 set where sample i is a case; sex_counts is [n_perm][2], the male
 * (sex == 1) and female cases.  Any ncase from 0 to N is drawn; n_perm == 0: DNAF_E_ARG.  Synchronous.
 */
int dnaf_perm_case_masks(dnaf_ctx* ctx, uint64_t seed, uint64_t first_perm, uint32_t n_perm, uint32_t* masks,
                         uint32_t* sex_counts);
/*
 * max(T) permutation tests of rows [row_begin,row_end) under permutations 0 .. n_perm - 1: t_obs is [rows][2], the
 * observed ALLELIC (the .assoc CHISQ, haploid cells included) and REC (2x2 Pearson n11 / n12 + n22 over the diploid
 * cells, no cell rule) statistics, NaN where a denominator is 0 (no test; Y and MT rows have no REC).  exceed is
 * [rows][2], the permutations whose statistic T_p >= T_obs (1 - 1e-7); max_t is [n_perm][2], the maximum of T_p over
 * the rows with a test (0 where none has one).  Under permutation p the case margins follow from the row class and
 * p's male and female cases (m, f): case alleles 2(m + f), 2f + m, m, m + f and case diploid cells m + f, f, 0, 0 on
 * autosome, X, Y, MT rows; the row totals are those of dnaf_genotype_counts.  EMP1 = (exceed + 1) / (n_perm + 1),
 * EMP2 = (#{p : max_t[p] >= T_obs (1 - 1e-7)} + 1) / (n_perm + 1).  max_t composes over row ranges by elementwise max.
 * Rows with more than 2 alleles: DNAF_E_INPUT before any GPU work, naming the row; no cases, no controls or
 * n_perm == 0: DNAF_E_ARG.
 */
int dnaf_mperm(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t n_perm, double* t_obs,
               uint32_t* exceed, double* max_t, dnaf_stats* stats);
/* Same work, results left in device memory. */
int dnaf_mperm_device(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint32_t n_perm,
                      dnaf_stats* stats);
/*
 * The .mperm body lines of n rows (PLINK 1.9's plink.assoc.mperm: CHR SNP EMP1 EMP2; labels as in dnaf_format_assoc):
 * emp is [n][2] (EMP1, EMP2), printed "%.4g", NA for NaN.  `out` holds at least 96 bytes per row.  Returns the bytes
 * written.
 */
uint64_t dnaf_format_mperm(uint64_t n, const int32_t* chrom_idx, const char* labels, const int64_t* ids, const double* emp,
                           char* out);

/* Parity gates. genotypes: out[(r*n_samples+i)*2+s] = allele index, 0xFF where the cell has no such
 * allele (second slot of a haploid cell, both slots of '.').  text: the uncompressed rows. */
int dnaf_genotypes(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint8_t* out,
                   uint64_t out_cap);
int dnaf_text(dnaf_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint64_t seed, uint8_t* out, uint64_t out_cap,
              uint64_t* n_bytes);

/* BgzfWriter.write() for arbitrary bytes (used for the VCF header, pop_factory.py:404-405, and the .tbi payload):
 * cuts `text` every 65280 bytes and encodes each piece on the GPU with the generic encoder (byte-4-back parse,
 * per-block dynamic Huffman).  It has one parse, so it takes no level (ABI 4 accepted and ignored one).  No EOF block. */
int dnaf_bgzf_compress(dnaf_ctx* ctx, const uint8_t* text, uint64_t n_bytes, uint8_t* out,
                       uint64_t out_cap, dnaf_stats* stats);
uint64_t dnaf_bgzf_bound(uint64_t text_bytes);
/* Block table of a BGZF stream held in host memory (no GPU work, no context): compressed and text size of
 * every block, in order.  With csize == usize == NULL only counts.  DNAF_E_INPUT when the bytes are not a
 * whole number of well-formed BGZF blocks, DNAF_E_SPACE when there are more than `cap` (n_blocks is still set).
 * This is what a tabix index needs besides the row sizes: virtual offset = block start << 16 | offset in block
 * (SURVEY 8f-3; the reference leaves indexing to `bcftools index`, README.md:98-99). */
int dnaf_bgzf_scan(const uint8_t* data, uint64_t n_bytes, uint32_t* csize, uint32_t* usize, uint64_t cap,
                   uint64_t* n_blocks);
/* The same table for streams that never reach the caller (dnaf_generate_fd) or reach it piecewise:
 * dnaf_block_log(ctx, 1) clears the log and makes every later dnaf_generate / _stream / _fd call append the
 * blocks it hands to the host; dnaf_block_log(ctx, 0) stops and clears.  The pointers returned by
 * dnaf_block_log_get stay valid until the next dnaf_generate* / dnaf_block_log call on the context. */
int dnaf_block_log(dnaf_ctx* ctx, int enable);
int dnaf_block_log_get(dnaf_ctx* ctx, const uint32_t** csize, const uint32_t** usize, uint64_t* n_blocks);
/* Self-test hook of the LZ tiers (-z 4..9; csrc/k_lz.cuh): host code, no context, no GPU.  Encodes ONE autosome
 * segment -- n_cells cells given as allele bits (bit 2i / 2i+1 = first / second allele of cell i), with the row
 * prefix when prefix_len > 0, ending in '\n' when ends_row -- with the span grammar and the static code tables the
 * kernel uses for minor-allele probability p_minor, and returns the raw deflate bytes (or a negative DNAF_E_*).
 * It exists so that the CPU test suite can inflate what the table builder and the grammar produce; the product
 * path never calls it. */
int64_t dnaf_debug_lz_block(double p_minor, int level, const uint32_t* allele_bits, uint32_t n_cells, const uint8_t* prefix,
                            uint32_t prefix_len, int ends_row, uint8_t* out, uint64_t out_cap);
/* The 28-byte BGZF end-of-file block BgzfWriter.close() appends. */
int dnaf_bgzf_eof(uint8_t* out28);

#ifdef __cplusplus
}
#endif
#endif /* DNAF_B200_H */
