/* longsom_host.h -- C-ABI of liblongsom_host.so, the CPU-side BAM/TSV codec library next to the CUDA
 * library (include/longsom_b200.h).  No CUDA, no torch types: plain pointers and sizes.
 *
 * It replaces, for the hot path and the steps on either side of it, what the reference does through
 * pysam / htslib and Python string formatting:
 *   ls_bam_read ...........  pysam.AlignmentFile(bam) + per-record accessors
 *                            (SNVCalling/BaseCellCounter.py:190-191,225-262; CellClustering/SingleCellGenotype.py:123)
 *   ls_write_counter_rows .  the per-site row formatting of BaseCellCounter.run_interval (:297-309)
 *   ls_bam_split ..........  PreProcessing/SplitBamCellTypes.py:39-192 (fetch / filter / trim / write / pysam.index)
 * Binding: longsom_b200/bamio.py, pipeline.py, cli/splitbam.py (ctypes).
 */
#ifndef LONGSOM_HOST_H
#define LONGSOM_HOST_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- BAM -> structure-of-arrays (the layout of ls_read_batch in longsom_b200.h) ------------------- */
/* Inflates the whole BGZF file with `threads` workers and parses every record.  Always returns a
 * handle; ls_bam_error() is non-NULL when decoding failed.  CB:Z tags are interned: array 4 holds a
 * dense barcode id per read (-1 = no tag), ls_bam_barcode(i) the raw tag text. */
void *ls_bam_read(const char *path, int threads);
const char *ls_bam_error(void *h);
void ls_bam_free(void *h);
int64_t ls_bam_n_reads(void *h);
int64_t ls_bam_n_cigar(void *h);
int64_t ls_bam_n_bases(void *h);
int32_t ls_bam_n_contigs(void *h);
const char *ls_bam_contig_name(void *h, int i);
int32_t ls_bam_contig_len(void *h, int i);
int32_t ls_bam_n_barcodes(void *h);
const char *ls_bam_barcode(void *h, int i);
const char *ls_bam_header_text(void *h);
/* which: 0 tid(i32) 1 pos(i32) 2 flag(u16) 3 mapq(u8) 4 barcode id(i32) 5 cigar_off(u32, n+1) 6 cigar(u32)
 *        7 base_off(u64, n+1, multiples of 16) 8 l_qseq(i32) 9 seq4(u8, 2 bases/byte) 10 qual(u8) */
const void *ls_bam_array(void *h, int which);

/* ---- BaseCellCounter rows ---------------------------------------------------------------------- */
/* Appends (append != 0) or writes n rows "chrom\tpos+1\tref\tDP|NC|CC|BC|BQ|BCf|BCr\t..." to path;
 * counts = n x 26 words in the order of ls_site_counts.  Returns 0, -1 when the file cannot be opened. */
int ls_write_counter_rows(const char *path, const char *chrom, const int32_t *pos, const uint8_t *ref,
                          const uint32_t *counts, int64_t n, int threads, int append);

/* ---- streaming BAM decoder (bounded memory) ---------------------------------------------------------- */
/* The drop-in BaseCellCounter's reader (replaces the per-window pysam pileup fetches of BaseCellCounter.py:190-191,
 * 344-409): ls_bams_next() hands out the next ~target_bytes of inflated records (a record cut by the chunk end is
 * carried over) while a background thread already inflates and indexes the chunk after it; ls_bams_fill() copies the
 * current chunk into caller buffers (pinned staging memory) in the layout of ls_read_batch.  Barcode ids are stable
 * for the whole file; ls_bams_n_barcodes() is the table size when the CURRENT chunk was indexed.
 * ls_bams_next: number of records, 0 at end of file, -1 on error (ls_bams_error has the text). */
void *ls_bams_open(const char *path, int threads);
const char *ls_bams_error(void *h);
void ls_bams_close(void *h);
int32_t ls_bams_n_contigs(void *h);
const char *ls_bams_contig_name(void *h, int i);
int32_t ls_bams_contig_len(void *h, int i);
int32_t ls_bams_n_barcodes(void *h);
const char *ls_bams_barcode(void *h, int i);
/* Optional, after ls_bams_open and before the first ls_bams_next: the run only needs the records that overlap the n
 * regions [beg[i], end[i]) of reference tid[i] (0-based, any order; regions that touch are merged).  The reader then
 * reads and inflates only the BGZF members of the spans the BAM's .bai index lists for them (SAM spec 5.3), merged into
 * disjoint spans in file order, and hands out exactly the records of those spans: every record that overlaps a region,
 * and possibly others, in file order.  The index is <bam>.bai, else <bam without .bam>.bai; CSI is not read.
 * Returns 1 when the index is used; 0 when there is none or it is refused, and the whole file is read as without the
 * call: an index that cannot be parsed, whose reference count differs from the header's, that is older than the BAM
 * (mtime: a stale index could change the records a region gets), or one of whose offsets is past the end of the file
 * or not inside a BGZF member.  ls_bams_index_note() then gives the reason in one line (NULL while the index is used).
 * -1 when called after ls_bams_next or on a handle in error. */
int ls_bams_set_regions(void *h, int64_t n, const int32_t *tid, const int64_t *beg, const int64_t *end);
const char *ls_bams_index_note(void *h);
int64_t ls_bams_next(void *h, int64_t target_bytes, int64_t *n_cigar, int64_t *n_bases);
/* Compressed BGZF member bytes read and bytes inflated to produce the chunk the last ls_bams_next returned (the call that
 * returned 0 included).  With the index, the header's members are not counted; without it, they count in the first
 * chunk. */
void ls_bams_chunk_io(void *h, int64_t *compressed, int64_t *inflated);
int ls_bams_fill(void *h, int32_t *tid, int32_t *pos, uint16_t *flag, uint8_t *mapq, int32_t *cb, int32_t *l_qseq,
                 uint32_t *cigar_off, uint64_t *base_off, uint32_t *cigar, uint8_t *seq4, uint8_t *qual);
/* the same, plus ref_end[i] = pos + M/D/N/=/X lengths of read i (exclusive reference end; may be NULL) */
int ls_bams_fill2(void *h, int32_t *tid, int32_t *pos, uint16_t *flag, uint8_t *mapq, int32_t *cb, int32_t *l_qseq,
                  uint32_t *cigar_off, uint64_t *base_off, uint32_t *cigar, uint8_t *seq4, uint8_t *qual, int64_t *ref_end);
/* The decoders' own raw-DEFLATE inflater (RFC 1951, whole buffers, exact output size; ls_inflate.h): 1 if `in`
 * inflates to exactly out_len bytes, 0 otherwise (the readers then hand the member to zlib).  Exposed for tests. */
int ls_inflate_raw(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_len);

/* ---- MergeBaseCellCounts ------------------------------------------------------------------------------------ */
/* The lock-step cursor merge of MergeBaseCellCounts.py:116-204 over n (chrom, pos)-sorted BaseCellCounter tables: `header`
 * (date line, ##INFO lines, column names) is written first, n_header_lines (9) lines are skipped at the top of every
 * input.  Returns 0; 1 when a row is not "chrom<tab>integer<tab>ref<tab>info<tab>counts" (the caller then runs its Python
 * restatement, whose exceptions are the reference's); -1 on an I/O error (err). */
int ls_merge_tables(int32_t n, const char *const *paths, const char *out_path, const char *header, int32_t n_header_lines,
                    char *err, int32_t errlen);

/* ---- BaseCellCalling.step1: the per-row work ----------------------------------------------------------- */
/* Replaces the row loop of BaseCellCalling.step1.py:78-467 around the beta-binomial calls (which stay on the GPU, K2).
 * ls_s1_parse reads a byte range of the merged table (whole lines; "\n", "\r\n" and "\r" end a line; "##" lines are
 * copied through): ct_cols = the columns of the cell types.  It returns NULL with a message in err for any row the
 * reference would fail on -- the caller then runs its Python restatement on the range, whose exceptions are the
 * reference's.  Queries: q1 = (alt reads, depth) with alpha1/beta1, q2 = (alt cells, cells) with alpha2/beta2, in the
 * order the handle expects their ROUNDED tails back in ls_s1_format.  ls_s1_sites gives (contig id, POS) per row
 * (id -1 for a "##" line) for the reference-context lookup: ctx[row][11] = fetch(CHROM, POS-6, POS+5) upper-cased,
 * ctx_len[row] = bytes that exist, -1 = no context ('.').  --fisher_cutoff != 1 is not handled here.
 * `data` must stay valid until ls_s1_free; the text of ls_s1_format belongs to the handle. */
void *ls_s1_parse(const char *data, int64_t len, const int32_t *ct_cols, int32_t n_ct, int32_t min_reads,
                  int32_t min_cells, char *err, int32_t errlen);
void ls_s1_free(void *h);
int64_t ls_s1_n_rows(void *h);
int64_t ls_s1_n_data_rows(void *h);
int64_t ls_s1_n_q1(void *h);
int64_t ls_s1_n_q2(void *h);
void ls_s1_queries(void *h, int32_t *q1k, int32_t *q1n, int32_t *q2k, int32_t *q2n);
int32_t ls_s1_n_chroms(void *h);
const char *ls_s1_chrom(void *h, int32_t i);
void ls_s1_sites(void *h, int32_t *chrom, int64_t *pos);
int64_t ls_s1_format(void *h, const double *r1, const double *r2, const uint8_t *ctx, const int8_t *ctx_len,
                     const char *const *ct_names, int32_t min_ac_cells, int32_t min_ac_reads, int32_t min_cell_types,
                     int32_t max_cell_types, const char **text);

/* ---- SingleCellGenotype / HCCVSingleCellGenotype: the dense long table ------------------------------------ */
/* Expands the touched (site, cell) tuples of ls_genotype_sparse_* into the reference's rows, one per (site, barcode of
 * the metadata) -- SingleCellGenotype.py:128-214, HCCVSingleCellGenotype.py:126-212.  prefix[s]: the seven leading
 * columns of site s, tab-joined; index[s]: its INDEX column (NULL array when hccv); chrm[s]: the chrM shortcut applies;
 * the site's tuples are [hit_lo[s], hit_hi[s]) of the arrays, sorted by cell, p rounded to four places;
 * cell_text[c] = "barcode<tab>cell type".  Returns the text length (>= 0) and a malloc'd text (ls_geno_rows_free). */
int64_t ls_geno_rows(int32_t n_sites, const char *const *prefix, const char *const *index, const uint8_t *chrm,
                     const int64_t *hit_lo, const int64_t *hit_hi, const int32_t *t_cell, const int32_t *t_dp,
                     const int32_t *t_alt, const double *t_p, int32_t n_cells, const char *const *cell_text, int32_t hccv,
                     double pvalue, char **text);
void ls_geno_rows_free(char *text);

/* ---- BaseCellCalling.step2: site lists ------------------------------------------------------------------------ */
/* The editing / panel-of-normals lists of build_dict (BaseCellCalling.step2.py:197-221): tab separated, '#' comments,
 * columns chrom, pos.  ls_sitelist_read: 0 = parsed (handle in *h), 1 = a line the reference's loop would treat
 * differently (the caller runs its Python loop, which empties the list on any failure), -1 = unreadable file.
 * ls_sitelist_fill: per row the index of its chromosome name (ls_sitelist_chrom) and its position. */
int ls_sitelist_read(const char *path, void **h);
int64_t ls_sitelist_n(void *h);
int32_t ls_sitelist_n_chroms(void *h);
const char *ls_sitelist_chrom(void *h, int32_t i);
void ls_sitelist_fill(void *h, int32_t *chrom, int64_t *pos);
void ls_sitelist_free(void *h);

/* ---- SplitBamCellTypes --------------------------------------------------------------------------- */
/* Routes every placed record of the coordinate-sorted BAM in_path to out_paths[type of its barcode]
 * (+ ".bai" each).  Barcode table: n_bc keys, key i = bc_blob[bc_off[i] .. bc_off[i+1]), type bc_type[i];
 * the key of a read is its CB:Z text before the first '-'.  max_nm / max_nh < 0 and min_mapq <= 0 switch
 * the respective filter off; n_trim > 0 zeroes the base qualities of the read ends (soft clips extend the
 * trim; a clip of 20..29 bases counts as 30).  counters[36]: Total_reads, Pass_reads, CB_not_found,
 * CB_not_matched, then [4 + mask] = reads dropped for reason set mask (1 nM, 2 nM_not_found, 4 NH,
 * 8 NH_not_found, 16 MAPQ); first_seen[32]: 1-based ordinal of the first read dropped for that set.
 * Input and outputs are streamed (64 MB compressed input chunks, 16 MB of pending records per output).
 * Returns 0, or -1 with a message in err (errors the reference raises -- trim longer than a read, a read
 * without qualities, a non-string CB -- are reported, not skipped). */
int ls_bam_split(const char *in_path, int n_types, const char *const *out_paths, const char *bc_blob,
                 const uint32_t *bc_off, const int32_t *bc_type, int64_t n_bc, int min_mapq, int max_nm, int max_nh,
                 int n_trim, int threads, int level, int64_t *counters, int64_t *first_seen, char *err, int errlen);

#ifdef __cplusplus
}
#endif
#endif
