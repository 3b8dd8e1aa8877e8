/*
 * vf_ingest.h — C ABI of libvf_ingest.so: host ingest for stage 1 (SURVEY §8f rank 1).
 *
 * The reference never parses a genome or a VCF itself: per window it spawns
 * `samtools faidx | bcftools consensus` (utils/data_process.py:27,40-59,404,416-435), i.e. htslib does the
 * BGZF inflation and the text parsing, once per window.  Here both files are read ONCE: the FASTA becomes the
 * byte-per-base arrays that stage1.Genome uploads to HBM, one sample of the VCF becomes the sorted
 * structure-of-arrays that stage1.SampleVariants uploads (pos, ref_len, alt_off, alt_len, gt, alt_pool — the layout
 * vf_encode_windows consumes, include/vf_b200.h).
 *
 * Plain text, gzip and BGZF (.gz written by bgzip: concatenated gzip members with a 'BC' extra field) are accepted;
 * BGZF members are inflated in parallel.  Genotype semantics (= oracle/ingest_py.py, which restates them in Python):
 *   - records whose first called ALT is symbolic (<...>) or '*' are dropped (bcftools `-e 'ALT~"<.*>"'`);
 *   - hom-ref and missing genotypes are dropped; haploid calls count as homozygous;
 *   - a/a with a > 0 -> gt 2 (hom-alt) with ALT a; a het between two different single-base ALTs of a single-base REF
 *     -> gt 2 with the IUPAC code of the two ALTs; every other het -> gt 1 with the first called ALT;
 *   - per chromosome the records are stably sorted by position (0-based).
 *
 * Every function returns NULL / a negative value on error; vf_ingest_last_error() returns a thread-local message.
 * Handles own their memory until *_close; *_copy fill caller-owned buffers.
 */
#ifndef VF_INGEST_H
#define VF_INGEST_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* vf_ingest_last_error(void);

typedef struct vf_fasta vf_fasta;
/* Parse a whole FASTA.  n_threads <= 0: one per hardware thread. */
vf_fasta* vf_fasta_open(const char* path, int n_threads);
int vf_fasta_num_seqs(const vf_fasta* f);
const char* vf_fasta_name(const vf_fasta* f, int i);          /* first word after '>' */
int64_t vf_fasta_length(const vf_fasta* f, int i);
/* Copy sequence i (case preserved, line breaks removed) into dst[cap]; returns the length or -1. */
int64_t vf_fasta_copy(const vf_fasta* f, int i, uint8_t* dst, int64_t cap);
void vf_fasta_close(vf_fasta* f);

typedef struct vf_vcf vf_vcf;
/* Parse one sample's genotypes of a VCF.  sample == NULL: the first sample column. */
vf_vcf* vf_vcf_open(const char* path, const char* sample, int n_threads);
int vf_vcf_num_chroms(const vf_vcf* v);
const char* vf_vcf_chrom(const vf_vcf* v, int c);
int64_t vf_vcf_num_records(const vf_vcf* v, int c);
int64_t vf_vcf_alt_bytes(const vf_vcf* v, int c);
/* Fill caller arrays of vf_vcf_num_records(c) entries (alt_pool: vf_vcf_alt_bytes(c) bytes).  Returns 0 or -1. */
int vf_vcf_copy(const vf_vcf* v, int c, int64_t* pos, int32_t* ref_len, int32_t* alt_off, int32_t* alt_len,
                uint8_t* gt, uint8_t* alt_pool);
void vf_vcf_close(vf_vcf* v);

typedef struct vf_vcf_cohort vf_vcf_cohort;
/* Parse many samples of a VCF in one pass: each data line is split once and every requested sample column decoded
 * from it with vf_vcf_open's genotype rules, so sample s's arrays of a chromosome equal what vf_vcf_open(path,
 * samples[s]) + vf_vcf_copy give (a chromosome where s keeps no record has 0 records).
 * samples == NULL: every sample column of the '#CHROM' line, in file order (n_samples is ignored).  An unknown or a
 * twice-requested sample fails, and so does a file without sample columns (a sites-only VCF).  regions_bed: NULL, or BED text ("chrom<TAB>start<TAB>end" lines, 0-based half-open;
 * '#', 'track' and 'browser' lines skipped): only records whose REF span [pos, pos + max(ref_len, 1)) intersects an
 * interval are kept, before any genotype is decoded. */
vf_vcf_cohort* vf_vcf_open_cohort(const char* path, const char* const* samples, int n_samples, const char* regions_bed,
                                  int n_threads);
int vf_vcf_cohort_num_samples(const vf_vcf_cohort* v);
const char* vf_vcf_cohort_sample_name(const vf_vcf_cohort* v, int s);
int vf_vcf_cohort_num_chroms(const vf_vcf_cohort* v);           /* chromosomes with a kept record of any sample */
const char* vf_vcf_cohort_chrom(const vf_vcf_cohort* v, int c);
int64_t vf_vcf_cohort_num_records(const vf_vcf_cohort* v, int s, int c);
int64_t vf_vcf_cohort_alt_bytes(const vf_vcf_cohort* v, int s, int c);
/* vf_vcf_copy's arrays of sample s, chromosome c.  Returns 0 or -1. */
int vf_vcf_cohort_copy(const vf_vcf_cohort* v, int s, int c, int64_t* pos, int32_t* ref_len, int32_t* alt_off,
                       int32_t* alt_len, uint8_t* gt, uint8_t* alt_pool);
void vf_vcf_cohort_close(vf_vcf_cohort* v);

#ifdef __cplusplus
}
#endif
#endif /* VF_INGEST_H */
