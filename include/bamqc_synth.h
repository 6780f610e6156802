/* bamqc_synth.h -- seeded synthetic BAM/FASTA generator (C ABI).
 *
 * The reference ships no fixtures (SURVEY.md section 4), so every test and benchmark input is produced
 * by this generator (SURVEY.md section 8d: standard 2x150 bp paired-end record, 290 B inflated).
 * It is tooling around the hot path, not part of the drop-in boundary (that is bamqc_b200.h).
 *
 * Reference genome bases are iid uniform ACGT, stored 2-bit packed: base i of a contig lives in
 * byte i/4, bits 2*(i%4) (A=0 C=1 G=2 T=3) -- the layout bqc_set_reference() expects.
 */
#ifndef BAMQC_SYNTH_H_
#define BAMQC_SYNTH_H_
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct bqc_synth_params {
    uint64_t seed;
    int32_t n_contigs;            /* contigs of the genome (all appear in the BAM header) */
    const char* const* names;     /* n_contigs names */
    const uint64_t* lengths;      /* n_contigs lengths */
    const uint8_t* const* packed; /* n_contigs 2-bit packed sequences (bqc_synth_reference) */
    const uint64_t* region_begin; /* optional per contig: fragments start in [begin,end); NULL = whole contig */
    const uint64_t* region_end;
    uint64_t n_pairs;             /* target number of primary pairs in the regions (approximate, +-0.5%) */
    int32_t read_len;             /* 150 */
    double ins_mean, ins_sd;      /* insert size ~ round(N(mean, sd)) clamped to [ins_min, ins_max] */
    int32_t ins_min, ins_max;
    double sub_rate;              /* per-base substitution rate (0.005) */
    double n_rate;                /* per-base N rate in reads (0.001) */
    double indel_read_frac;       /* fraction of mapped reads with indels (0.03) */
    int32_t max_indels;           /* 1 (stress: 3) */
    double softclip_frac;         /* fraction of mapped reads soft-clipped (0.03) */
    int32_t low_quality;          /* 0 = standard quality profile, 1 = mean ~Q15 (cfg 4) */
    double mapq60_frac;           /* 0.9; stress: -1 => uniform 0..60 */
    double dup_frac, qcfail_frac; /* per pair: 0.02, 0.005 */
    double one_unmapped_frac;     /* 0.01 */
    double both_unmapped_frac;    /* 0.005 (emitted at the end, rID -1) */
    double secondary_frac, supplementary_frac; /* extra records: 0.005 each */
    int32_t n_lanes;              /* read groups L1..Ln, assigned per pair uniformly */
    uint64_t first_pair_id;       /* read names are p%09llu starting here (shards use disjoint ranges) */
    int32_t emit_unmapped_tail;   /* 1 = append the both-unmapped pairs of this shard */
} bqc_synth_params;

/* Fill *p with the SURVEY section 8(d) defaults (cfg 1/2 library). */
void bqc_synth_default_params(bqc_synth_params* p);

/* Deterministic contig sequence for (seed, contig_index): writes (n_bases+3)/4 bytes (rounded up to 8). */
void bqc_synth_reference(uint64_t seed, int32_t contig_index, uint64_t n_bases, uint8_t* packed_out);

/* 60-column FASTA of the packed contigs. Returns 0 on success. */
int bqc_synth_write_fasta(const char* path, int32_t n_contigs, const char* const* names,
                          const uint64_t* lengths, const uint8_t* const* packed);

/* SAM header text (@HD, @SQ.., @RG..) for the params; returns length, writes at most cap bytes. */
size_t bqc_synth_header_text(const bqc_synth_params* p, const char* sample_id, char* out, size_t cap);

/* Generate coordinate-sorted inflated BAM records (block_size prefix included) into `out`.
 * offsets_out receives n_records+1 byte offsets. Returns 0 on success, 1 if a capacity was too small
 * (then *n_bytes / *n_records hold what would have been needed so far). */
int bqc_synth_records(const bqc_synth_params* p, uint8_t* out, uint64_t out_cap, uint64_t* n_bytes,
                      uint64_t* offsets_out, uint64_t offsets_cap, uint64_t* n_records);

/* Write a complete BAM file: header + records. compress_level 0..9 => BGZF (deflate level; 0 = stored
 * blocks); -1 => raw uncompressed BAM byte stream (no BGZF container). Returns 0 on success. */
int bqc_synth_write_bam(const char* path, const bqc_synth_params* p, const char* sample_id,
                        const uint8_t* records, uint64_t n_bytes, int compress_level);

/* Write a SAM text file: the header of bqc_synth_header_text and one alignment line per record. Returns 0 on success. */
int bqc_synth_write_sam(const char* path, const bqc_synth_params* p, const char* sample_id, const uint8_t* records, uint64_t n_bytes);

/* BGZF-compress an arbitrary byte stream into memory (for end-to-end inflate benchmarks).
 * Returns compressed size, or 0 if cap is too small. */
uint64_t bqc_synth_bgzf_compress(const uint8_t* in, uint64_t n, int level, uint8_t* out, uint64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* BAMQC_SYNTH_H_ */
