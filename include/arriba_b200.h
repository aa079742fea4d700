/* arriba_b200.h -- C ABI of the B200-native implementation of Arriba's post-alignment hot path.
 *
 * The reference (suhrig/arriba v2.5.1) has no FFI: its seam is the set of C++ free functions that
 * `main` (source/arriba.cpp:79) calls on two in-memory containers. Each entry point below names the
 * reference function(s) it replaces. Plain pointers and sizes only; all arrays are caller-owned host
 * memory (pinned memory makes the copies asynchronous), device memory is library-owned.
 * Every function returns 0 on success, non-zero on error (message via arb_last_error). No exceptions
 * cross the boundary. One context per thread; a context is bound to one CUDA device.
 * There is no CPU fallback: arb_ctx_create fails when no CUDA device is usable.
 */
#ifndef ARRIBA_B200_H
#define ARRIBA_B200_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ARB_N_FILTERS 38 /* filter ids follow the reference registry, source/common.hpp:30-67 */

typedef struct arb_ctx arb_ctx;

int arb_ctx_create(arb_ctx** out, int device);
void arb_ctx_destroy(arb_ctx* ctx);
const char* arb_last_error(arb_ctx* ctx);         /* ctx may be NULL: last error of arb_ctx_create */
const char* arb_backend(void);                    /* "cuda-sm_100a" for the product library */
uint64_t arb_kernel_launches(void);               /* kernels launched by this library since load */
/* sizeof() of the public structs, for bindings to verify their layout: arb_contigs, arb_annotation, arb_params, arb_soa_chunk, arb_candidates,
   arb_evalue_inputs, arb_timings, arb_run_options, arb_run_stats */
void arb_struct_sizes(uint32_t out[9]);

/* ---- reference genome and annotation --------------------------------------------------------------------
 * Replaces the in-memory products of load_assembly (source/assembly.cpp:28), read_annotation_gtf
 * (source/annotation.cpp:161) and make_annotation_index (source/annotation.t.hpp:25) as inputs of the kernels. */
typedef struct arb_contigs {
	uint32_t n_contigs;
	const uint8_t* flags;          /* bit0 interesting (-i), bit1 viral (-v) */
	const uint32_t* length;        /* 0 if the sequence is not loaded */
	const char* const* sequence;   /* upper-case bases per contig, NULL if not loaded */
} arb_contigs;
int arb_set_contigs(arb_ctx* ctx, const arb_contigs* contigs);
/* per-sample contig flags without re-sending the sequences: bit0 interesting, bit1 viral, bit2 / bit3 = verdicts of filter_top_expressed_viral_contigs /
   filter_low_coverage_viral_contigs on a viral contig (computed by the caller per contig; the per-fragment rules run in arb_run_read_filters) */
int arb_set_contig_flags(arb_ctx* ctx, const uint8_t* flags, uint32_t n_contigs);

typedef struct arb_annotation {
	uint32_t n_genes;              /* gene id == index; ids ascend in creation order (GTF order, then dummy genes) */
	const uint16_t* gene_contig; const int32_t* gene_start; const int32_t* gene_end;
	const uint8_t* gene_strand;    /* 1 = forward */
	const int32_t* gene_exonic_length;
	const uint8_t* gene_flags;     /* bit0 dummy, bit1 protein coding */
	uint32_t n_exons;              /* exon id == index, creation (GTF) order */
	const uint32_t* exon_gene; const int32_t* exon_start; const int32_t* exon_end;
	const int32_t* exon_cds_start; const int32_t* exon_cds_end; /* -1 = none */
	const int32_t* exon_next_start;                             /* start of the next exon of the transcript, -1 = none */
	const uint8_t* exon_flags;     /* bit0 has previous exon, bit1 has next exon */
	uint32_t n_contigs;
	/* disjoint-region indices: region r of contig c (exon_region_begin[c] <= r < exon_region_begin[c+1]) covers
	   (end[r-1], end[r]] and lists the ids overlapping it (ascending) */
	const uint32_t* exon_region_begin; const int32_t* exon_region_end; const uint32_t* exon_region_off; const uint32_t* exon_region_items;
	const uint32_t* gene_region_begin; const int32_t* gene_region_end; const uint32_t* gene_region_off; const uint32_t* gene_region_items;
} arb_annotation;
int arb_set_annotation(arb_ctx* ctx, const arb_annotation* annotation);

/* ---- options that the kernels need (subset of options_t, source/options.hpp:25-69; defaults options.cpp:71-107) */
typedef struct arb_params {
	uint64_t filter_mask;              /* bit f set = filter id f enabled (-f clears bits) */
	uint32_t homopolymer_length;       /* -H 6 */
	int32_t min_read_through_distance; /* -R 10000 */
	float max_kmer_content;            /* -K 0.6 */
	uint32_t max_itd_length;           /* -l 100 */
	uint32_t external_duplicate_marking; /* -u */
	float mismatch_pvalue_cutoff;      /* -V 0.01 */
	uint32_t subsampling_threshold;    /* -U 300 */
	float evalue_cutoff;               /* -E 0.3 */
	float max_mismapper_fraction;      /* -m 0.8 */
	float max_homolog_identity;        /* -L 0.3 */
} arb_params;
void arb_default_params(arb_params* p);
int arb_set_params(arb_ctx* ctx, const arb_params* p);

/* ---- fragments -----------------------------------------------------------------------------------------
 * Structure-of-arrays image of chimeric_alignments_t (source/common.hpp:191-220) as produced by
 * read_chimeric_alignments (source/read_chimeric_alignments.cpp:560) + annotation (arriba.cpp:165-325).
 * Fragments are in NAME ORDER of "<qname>,<HI>" (the std::map order every reference loop relies on);
 * the index of a fragment is its name rank. Per-alignment arrays hold 3*n entries: index = slot*n + fragment,
 * slot 0 = MATE1, 1 = MATE2 / SPLIT_READ, 2 = SUPPLEMENTARY (unused for discordant mates). */
typedef struct arb_soa_chunk {
	uint32_t n_fragments;
	const uint8_t* n_aln;          /* 2 or 3 */
	const uint8_t* fflags;         /* bit0 single_end, bit1 multimapper, bit2 duplicate (BAM 0x400), bit3 same read name (up to the last comma) as the fragment before */
	const uint8_t* filter;         /* initial labels (normally all 0) */
	const uint16_t* contig; const int32_t* start; const int32_t* end;
	const uint8_t* aflags;         /* bit0 supplementary, 1 first_in_pair, 2 exonic, 3 forward strand, 4 predicted strand forward, 5 predicted strand ambiguous */
	const uint32_t* cigar_off; const uint16_t* cigar_cnt;
	const uint32_t* seq_off;       /* slots 0 and 1 (2*n entries used), units of 16 bytes */
	const uint16_t* seq_len;
	const uint32_t* genes_off; const uint16_t* genes_cnt;
	const uint32_t* cigar; uint64_t n_cigar;     /* BAM-encoded CIGAR operations */
	const uint8_t* seq; uint64_t n_seq_bytes;    /* nt16 4-bit bases, BAM nibble order */
	const uint32_t* genes; uint64_t n_genes;     /* gene ids, each set ascending */
} arb_soa_chunk;
int arb_push_chunk(arb_ctx* ctx, const arb_soa_chunk* chunk); /* H2D copy; replaces the resident fragment table */
/* The same in two parts, so that the copy overlaps the caller's annotation pass: _begin copies everything read_chimeric_alignments produced (all columns but
 * aflags and the gene sets) asynchronously on the context's copy stream; _end copies aflags / genes_off / genes_cnt / genes and returns when the table is
 * resident. The columns must stay valid and unchanged (apart from the annotation columns) between the two calls. Copies are asynchronous when the columns
 * are page-locked; the whole-run driver builds them in page-locked blocks (cudaHostAlloc, recycled across samples). */
int arb_push_chunk_begin(arb_ctx* ctx, const arb_soa_chunk* chunk);
int arb_push_chunk_end(arb_ctx* ctx, const arb_soa_chunk* chunk);
/* ---- BAM records of an inflated chunk -------------------------------------------------------------------------
 * The bookkeeping the reference's record loop (source/read_chimeric_alignments.cpp:611, sam_read1) does implicitly: where the records of a chunk of inflated
 * BGZF payload start (SAMv1 4.2: every record begins with its block_size) and which worker parses which record -- lists by read-name hash (FNV-1a), so that
 * the records of a fragment meet in one list; file order is kept inside a list. chunk: page-locked host memory makes the copy asynchronous; first = offset of
 * the first record; n_ref = reference sequences of the BAM header (sanity of guessed record starts); consumed = offset behind the last complete record;
 * record_offsets: capacity bytes / 36 + 1; malformed != 0: a block_size < 33 was met where a one-thread walk would have met it. */
int arb_bam_scan(arb_ctx* ctx, const uint8_t* chunk, uint64_t bytes, uint64_t first, int32_t n_ref, uint32_t n_lists, uint64_t* consumed, uint32_t* n_records,
                 uint32_t* list_begin /* n_lists + 1 */, uint32_t* record_offsets, uint32_t* malformed);
/* ---- the fragment table, built on the device from the ingest workers' pools ---------------------------------------
 * The end of read_chimeric_alignments (source/read_chimeric_alignments.cpp:340-506 slot normalisation and rejection of malformed fragments, the std::map
 * order of "<qname>,<HI>[ITD]", :792-802 mark_multimappers). Every worker of the record loop owns append-only pools: read names, CIGAR operations, nt16
 * sequences (each 16-byte aligned), alignments (linked per fragment through `next`, worker-local indices) and fragments (`head` = first alignment; offsets
 * into the worker's own pools). arb_build_fragment_table copies the pools to the device and leaves the fragment table resident in name order, as
 * arb_push_chunk_begin would (the annotation columns follow through arb_annotate_pass1/2). arb_get_fragment_table copies it back into caller columns sized
 * from `sizes`: 3*n per slot column (seq_off / seq_len 2*n), n_cigar, n_seq_bytes, n_name_bytes, n + 1 name offsets. Names of one table must be unique. */
typedef struct arb_pool_alignment { uint8_t supplementary, first_in_pair, forward; uint16_t contig; int32_t start, end; uint32_t cigar_off, cigar_cnt; uint64_t seq_off; uint32_t seq_len; int32_t next; } arb_pool_alignment;
typedef struct arb_pool_fragment { uint64_t name_off; uint32_t name_len; int32_t head, tail; uint32_t count; uint8_t single_end, duplicate; } arb_pool_fragment;
typedef struct arb_ingest_pool {
	const char* names; uint64_t n_name_bytes; const uint32_t* cigars; uint64_t n_cigars; const uint8_t* seqs; uint64_t n_seq_bytes;
	const arb_pool_alignment* alns; uint64_t n_alns; const arb_pool_fragment* frags; uint32_t n_frags;
} arb_ingest_pool;
typedef struct arb_fragment_table_sizes {
	uint32_t n_fragments;  /* fragments that survived slot normalisation */
	uint32_t tie_rounds;   /* rounds of the name sort beyond the first 16 bytes of the names */
	uint64_t n_rejected;   /* malformed fragments (the reference's "malformed SAM records" warning counts them) */
	uint64_t n_cigar, n_seq_bytes, n_name_bytes;
	float upload_ms, build_ms;  /* copy of the pools; the whole call (copy included), both on the context's stream */
} arb_fragment_table_sizes;
typedef struct arb_fragment_columns {
	uint8_t* n_aln; uint8_t* fflags; uint8_t* filter; uint16_t* contig; int32_t* start; int32_t* end; uint8_t* aflags; uint32_t* cigar_off; uint16_t* cigar_cnt;
	uint32_t* seq_off; uint16_t* seq_len; uint32_t* cigar; uint8_t* seq; char* names; uint64_t* name_off;
} arb_fragment_columns;
int arb_build_fragment_table(arb_ctx* ctx, const arb_ingest_pool* pools, uint32_t n_pools, arb_fragment_table_sizes* sizes);
int arb_get_fragment_table(arb_ctx* ctx, const arb_fragment_columns* out);
uint32_t arb_fragment_table_tie_rounds(arb_ctx* ctx); /* tie_rounds of the last arb_build_fragment_table */
/* ---- annotation of the resident fragments -------------------------------------------------------------------
 * Replaces the annotation passes of main (source/arriba.cpp:165-325: annotate_alignments per fragment, source/annotation.cpp:431-555; dummy genes for
 * intergenic breakpoints, arriba.cpp:207-260; second pass :262-319) and assign_strands_from_strandedness (source/read_chimeric_alignments.cpp:775-790).
 * Call sequence: arb_set_annotation (genes of the GTF) and arb_push_chunk_begin, then
 *   arb_annotate_pass1  : `aflags` = the alignment flags as ingest left them (3*n); strandedness 0 no, 1 yes, 2 reverse. Returns the number of dummy genes,
 *   arb_get_dummy_genes : their (contig, start, end) in creation order; the caller appends them to its gene table, rebuilds its gene index and
 *   arb_set_annotation  : sends the grown table, then
 *   arb_annotate_pass2  : finishes the gene sets; the resident table is complete (no arb_push_chunk_end). n_gene_ids = size of the gene-id pool,
 *   arb_get_annotation_columns : the annotation columns for host-side consumers (caller-allocated: 3*n, 3*n, 3*n, n_gene_ids). */
int arb_annotate_pass1(arb_ctx* ctx, const uint8_t* aflags, int32_t strandedness, uint32_t* n_dummy_genes);
int arb_get_dummy_genes(arb_ctx* ctx, uint16_t* contig, int32_t* start, int32_t* end);
int arb_annotate_pass2(arb_ctx* ctx, uint64_t* n_gene_ids);
int arb_get_annotation_columns(arb_ctx* ctx, uint8_t* aflags, uint32_t* genes_off, uint16_t* genes_cnt, uint32_t* genes);
void arb_set_host_memory_device(int device); /* device whose context page-locks the host blocks (one process per GPU: the process's device) */

/* ---- read-level filter cascade ---------------------------------------------------------------------------
 * Replaces filter_duplicates, filter_uninteresting_contigs, filter_viral_contigs, filter_proximal_read_through,
 * filter_inconsistently_clipped_mates, filter_homopolymer, filter_small_insert_size, filter_long_gap, filter_same_gene,
 * filter_hairpin, filter_mismatches, filter_low_entropy (source/filter_*.cpp; call order arriba.cpp:327-409).
 * genome_size: sum of the lengths of interesting contigs (filter_mismatches.cpp:105-108). */
int arb_run_read_filters(arb_ctx* ctx);
int arb_get_fragment_filters(arb_ctx* ctx, uint8_t* filter_out /* n */, uint8_t* early_out /* n or NULL: labels after the contig filters */);
int arb_set_fragment_filters(arb_ctx* ctx, const uint8_t* filter /* n */); /* host-side filters (viral, multimappers, ITD recovery) write back */
int arb_get_filter_counts(arb_ctx* ctx, uint32_t counts[ARB_N_FILTERS]); /* fragments per label; `(remaining=..)` lines derive from it */

/* ---- candidate generation --------------------------------------------------------------------------------
 * Replaces find_fusions (source/fusions.cpp:203). Candidates are numbered in the order the reference would first
 * insert them into fusions_t (fragment name order, then gene1 x gene2 loop order). */
typedef struct arb_candidates {
	uint32_t n;
	uint32_t *gene1, *gene2; uint16_t *contig1, *contig2; int32_t *breakpoint1, *breakpoint2; uint8_t *direction1, *direction2; /* 1 = upstream */
	uint32_t *split_reads1, *split_reads2, *discordant_mates;
	uint8_t* filter;
	uint8_t* bits;   /* 1 exonic1, 2 exonic2, 4 spliced1, 8 spliced2, 16 predicted_strand1 fwd, 32 predicted_strand2 fwd, 64 predicted strands ambiguous,
	                    128 transcript start = gene1 */
	uint8_t* bits2;  /* 1 transcript start ambiguous */
	int32_t *anchor_start1, *anchor_start2;
	float* evalue;
	uint32_t *list1_off, *list2_off, *listd_off; /* n+1 each */
	uint32_t *list1, *list2, *listd;             /* fragment indices (name ranks), name order */
} arb_candidates;
int arb_find_fusions(arb_ctx* ctx, int32_t max_mate_gap);
int arb_candidates_size(arb_ctx* ctx, uint32_t* n, uint64_t* n_list1, uint64_t* n_list2, uint64_t* n_listd);
int arb_get_candidates(arb_ctx* ctx, arb_candidates* out /* caller-allocated to arb_candidates_size */);
/* Multi-GPU runs shard the fragments by contig pair (SURVEY.md section 8e): every rank finds the candidates of its shard, the tables are exchanged
 * and merged by (first fragment, local id) -- the order the reference would have inserted them -- and installed with arb_set_candidates. */
int arb_get_candidate_first_fragments(arb_ctx* ctx, uint32_t* first_fragment_out /* n candidates: fragment that created the candidate */);
int arb_set_candidates(arb_ctx* ctx, const arb_candidates* table); /* replaces the resident candidate table */
int arb_apply_slot_swaps(arb_ctx* ctx, const uint8_t* swapped /* n fragments */); /* canonical mate order of another rank's find_fusions */
int arb_get_slot_swaps(arb_ctx* ctx, uint8_t* swapped_out /* n fragments: 1 if MATE1/MATE2 were canonicalised (fusions.cpp:416-421) */);

/* ---- event-level stages on the candidate table ------------------------------------------------------------------
 * The mutable candidate columns (filter, read counts, e-value) travel between the host-side event logic and the device
 * with arb_set/get_candidate_state; candidates are addressed by their id (first-insertion order). */
int arb_set_candidate_state(arb_ctx* ctx, const uint8_t* filter, const uint32_t* split_reads1, const uint32_t* split_reads2, const uint32_t* discordant_mates, const float* evalue);
int arb_get_candidate_filters(arb_ctx* ctx, uint8_t* filter /* n candidates */); /* the label column alone */
int arb_get_candidate_state(arb_ctx* ctx, uint8_t* filter, uint32_t* split_reads1, uint32_t* split_reads2, uint32_t* discordant_mates, float* evalue);
int arb_set_candidate_lists(arb_ctx* ctx, const uint32_t* list1_off, const uint32_t* list1, const uint32_t* list2_off, const uint32_t* list2);
/* Replaces merge_adjacent_fusions (source/merge_adjacent_fusions.cpp:19). n_itd_merges: internal tandem duplications whose read
 * lists must be concatenated by the caller; arb_get_merge_log returns (winner id, absorbed id, order key) triples. */
int arb_merge_adjacent(arb_ctx* ctx, int32_t max_distance, uint32_t* n_itd_merges);
int arb_get_merge_log(arb_ctx* ctx, uint32_t* triples /* 3*n */, uint32_t n);
/* Replaces the per-candidate part of estimate_expected_fusions (source/filter_relative_support.cpp:130-206); the order-dependent
 * global tallies (:19-127) and the pow() tables come from the caller so that the result is bit-identical to the reference's float. */
typedef struct arb_evalue_inputs {
	const int32_t* partner_count; uint32_t n_genes;
	uint32_t spliced_breakpoints, exonic_breakpoints, intronic_breakpoints, exonic_intronic_breakpoints;
	uint32_t intragenic_duplications, intragenic_inversions, spliced_same_gene, spliced_different_genes;
	float read_through_fraction; uint64_t mapped_reads;
	const double *pow_reads, *pow_intragenic, *pow_intergenic; uint32_t n_read_table;
	const double *pow_spliced1000 /* 1000 */, *pow_spliced400 /* 400 */, *pow_read_through /* 400000 */, *pow_proximal /* 400000 */;
	double read_through_penalty;
} arb_evalue_inputs;
int arb_estimate_evalues(arb_ctx* ctx, const arb_evalue_inputs* in);
int arb_filter_relative_support(arb_ctx* ctx, float evalue_cutoff); /* source/filter_relative_support.cpp:209 */
/* Replaces select_best (source/select_best.cpp): among the unfiltered candidates of one (gene1, gene2, direction1, direction2) the best one stays, visited in the
 * reference's iteration order (arb_replay_insertion_order must have run); *remaining = candidates still unfiltered */
int arb_select_best(arb_ctx* ctx, uint32_t* remaining);
/* global tallies of the e-value model over the resident candidate state (source/filter_relative_support.cpp:62-127), in this order: breakpoints of distant
 * fusions that are spliced / both exonic / both intronic / mixed, intragenic duplications, intragenic inversions, both-spliced candidates within one gene / between
 * two genes, genes with fusions, genes with read-through fusions, largest number of supporting reads of a candidate */
int arb_evalue_tallies(arb_ctx* ctx, uint32_t out[11]);
/* the per-candidate predicates between the e-value and its cutoff, on the resident candidate state: stage 0 = filter_non_coding_neighbors
 * (source/filter_non_coding_neighbors.cpp), 1 = filter_intragenic_both_exonic (source/filter_intragenic_both_exonic.cpp, -e exonic_fraction),
 * 2 = filter_min_support (source/filter_min_support.cpp, -S min_support); *remaining = candidates still unfiltered, the function's return value in the reference */
int arb_filter_simple(arb_ctx* ctx, int32_t stage, float exonic_fraction, int32_t min_support, uint32_t* remaining);

/* The order in which the reference's loops visit the candidates = the iteration order of fusions_t, a std::unordered_map (source/common.hpp:286-314) the
 * candidates were inserted into in id order; estimate_expected_fusions, select_best, recover_isoforms, filter_homologs and the discarded file depend on it.
 * libstdc++ puts a new node at the front of its bucket's run of the node list (a new bucket's run at the front of the list) and re-inserts the list, in
 * order, when the table grows: the order follows from a chain of sorts, one per growth, done on the device over the resident candidate keys. The growth
 * schedule is the caller's (its C++ library's std::__detail::_Prime_rehash_policy): candidates [phase_start[j], phase_start[j+1]) are inserted while the
 * table has phase_buckets[j] buckets; phase_start has n_phases + 1 entries. order_out[q] = id of the candidate visited q-th, rank_out = its inverse. */
int arb_replay_insertion_order(arb_ctx* ctx, const uint32_t* phase_start, const uint64_t* phase_buckets, uint32_t n_phases, uint32_t* order_out, uint32_t* rank_out);
/* Replaces the fusion-partner tally of estimate_expected_fusions (source/filter_relative_support.cpp:19-60) on the resident candidate state: of the
 * candidates that share (gene, breakpoint1, breakpoint2) only the first in the iteration order (arb_replay_insertion_order) contributes its partner;
 * partner_count_out[g] = distinct partners of g that have no more partners than g -- the `partner_count` input of arb_estimate_evalues. */
int arb_partner_counts(arb_ctx* ctx, int32_t* partner_count_out /* n_genes */);
/* Replaces filter_multimappers (source/filter_multimappers.cpp:115): of the fragments that share a read name (fflags bit1 / bit3) only the one with the best
 * alignment score keeps its label, ties go to the fragment whose best candidate has more support; read counts of the candidates follow. Works on the
 * resident candidate state and fragment labels; results through arb_get_candidate_state / arb_get_fragment_filters. */
int arb_filter_multimappers(arb_ctx* ctx);
/* Replaces find_top_expressed_genes' counting (source/filter_in_vitro.cpp:48-83) and the per-candidate verdicts of filter_in_vitro_generated_fusions
 * (:85-228). arb_set_coverage: the sample's coverage windows (source/read_stats.cpp:268-306: 20 bp windows per contig, n_windows[c] = 0 for contigs
 * without one). arb_reads_by_gene: supporting fragments per gene (the caller derives the expression quantile, -Q). arb_filter_in_vitro works on the
 * resident candidate state (arb_set_candidate_state) and fragment labels (arb_set_fragment_filters) and marks candidates F_in_vitro; exonic_pairs: sorted
 * (gene << 32 | partner) keys, one per exonic, unspliced breakpoint pair and direction (:93-104). */
int arb_set_coverage(arb_ctx* ctx, const uint16_t* const* coverage_per_contig, const uint64_t* n_windows, uint32_t n_contigs);
int arb_reads_by_gene(arb_ctx* ctx, uint32_t* reads_out /* n_genes */);
int arb_filter_in_vitro(arb_ctx* ctx, const uint32_t* reads_by_gene, uint32_t n_genes, uint32_t threshold, const uint64_t* exonic_pairs, uint64_t n_pairs);
/* spliced support of every candidate that may back another one up (source/recover_both_spliced.cpp:15-62, :104-118): support_out[k] = the support,
 * 0xFFFFFFFF where the candidate is not eligible or has none; works on the resident candidate state and fragment labels like arb_filter_in_vitro */
int arb_spliced_support(arb_ctx* ctx, const uint32_t* reads_by_gene, uint32_t n_genes, uint32_t threshold, uint32_t* support_out /* n candidates */);

/* ---- rows of the discarded-fusions file -------------------------------------------------------------------------------------
 * Replaces write_fusions_to_file (source/output_fusions.cpp:1043-1261) for the file of discarded fusions (-O) without -X: one row per candidate whose
 * filter is set, in the iteration order of the candidate map (arb_replay_insertion_order), formatted on the device from the resident candidate state,
 * fragment labels (filters column), annotation and coverage. The caller supplies what the device does not hold: names, the exons' neighbours in their
 * transcripts, the alphabetical order of the filter names, the confidence column. The header line stays with the caller. */
typedef struct arb_row_texts {
	uint32_t n_genes, n_exons, n_contigs;
	const char* gene_name; const uint32_t* gene_name_off;       /* string k = chars[off[k], off[k+1]) */
	const char* gene_id; const uint32_t* gene_id_off;
	const char* contig_name; const uint32_t* contig_name_off;   /* as named in the input files ("chr1") */
	const char* filter_name; const uint32_t* filter_name_off;   /* ARB_N_FILTERS names */
	const int32_t* exon_prev; const int32_t* exon_next;         /* exon ids, -1 = none */
	uint8_t filters_by_name[ARB_N_FILTERS];                     /* filter ids in alphabetical order of their names */
	uint32_t max_itd_length;
} arb_row_texts;
int arb_set_row_texts(arb_ctx* ctx, const arb_row_texts* texts);
int arb_format_discarded_rows(arb_ctx* ctx, const uint8_t* confidence /* per candidate: 0 low, 1 medium, 2 high */, uint64_t* n_rows, uint64_t* n_bytes);
int arb_get_row_text(arb_ctx* ctx, char* out /* n_bytes */);
/* ---- read pileups and consensus sequences of the rows of fusions.tsv ---------------------------------------------------------
 * arb_build_consensus replaces pileup_chimeric_alignments (source/output_fusions.cpp:25) and get_sequence_from_pileup (:109) as called by
 * get_fusion_transcript_sequence (:242-318) for a batch of candidates: per candidate two pileups (one per breakpoint) over ten views of its supporting reads,
 * each reduced to the consensus string, the genomic position of every character (-1 = none) and the bases beyond the breakpoint; and the number of
 * non-template bases between the fused segments (:300-318). Job 2 r + s is side s (0: breakpoint 1) of candidates[r]. arb_get_consensus copies the packed
 * results: *_off hold 2 n_rows + 1 offsets, verdict[j] != 0 marks a job the device left to the caller (tables full, 16-bit counters, empty insertion key),
 * non_template[r] == 0xFFFFFFFF a row whose non-template count the caller computes. Fragment labels and candidate state must be current on the device. */
typedef struct arb_consensus_info { uint32_t n_rows, retried_jobs; uint64_t seq_bytes, pos_count, clip_bytes; } arb_consensus_info;
int arb_build_consensus(arb_ctx* ctx, const uint32_t* candidates, uint32_t n_rows, arb_consensus_info* info);
int arb_get_consensus(arb_ctx* ctx, uint32_t* seq_off, uint32_t* pos_off, uint32_t* clip_off, uint8_t* verdict, uint32_t* non_template, char* seq, int32_t* pos, char* clip);

/* ---- k-mer index of the fused genes, gene homology, re-alignment of supporting reads -----------------------------------
 * arb_build_kmer_index replaces make_kmer_index (source/filter_mismappers.cpp:47): `intervals` are the disjoint, sorted unions of the
 * gene windows [start - padding, end + padding) per contig, as [start, end_exclusive) of positions whose 8-mer is indexed.
 * arb_homolog_pairs evaluates is_homolog (source/filter_homologs.cpp:13) for a batch of gene pairs; the order-dependent pairwise
 * resolution of filter_homologs (:65-141) stays with the caller. arb_filter_mismappers replaces filter_mismappers
 * (source/filter_mismappers.cpp:272); it needs current fragment labels (arb_set_fragment_filters) and candidate state. */
int arb_set_splice_sites(arb_ctx* ctx, const uint32_t* off /* n_genes+1 */, const int32_t* sites); /* downstream splice sites per gene, ascending */
int arb_build_kmer_index(arb_ctx* ctx, const uint32_t* contig, const int32_t* start, const int32_t* end_exclusive, uint32_t n_intervals, uint32_t n_index_contigs, uint64_t* n_indexed);
int arb_kmer_index_digest(arb_ctx* ctx, uint64_t* kmers, uint64_t* positions, uint64_t* checksum, uint32_t n_contigs); /* per contig; checksum = sum((kmer*1000003+pos)*0x9E3779B97F4A7C15) */
int arb_homolog_pairs(arb_ctx* ctx, const uint32_t* gene_a, const uint32_t* gene_b, uint32_t n, uint8_t* is_homolog_out);
int arb_filter_mismappers(arb_ctx* ctx, int32_t max_mate_gap, uint64_t* n_realigned);

/* ---- one sample on several GPUs (SURVEY.md section 8e; arriba_b200/csrc/exchange.cu, DESIGN.md section 7) --------------------------------------------
 * The library never communicates itself: it exposes DEVICE buffers, the caller moves them with its transport (NCCL through torch.distributed in
 * arriba_b200/sharded.py). The fragment table is replicated from the rank that ingested the BAM (broadcast over NVLink/NVSwitch), the work is divided:
 * arb_find_fusions only emits the breakpoints of the contig pairs the part owns, arb_filter_mismappers_part re-aligns every parts-th work item.
 *   exchange groups (broadcast): ARB_XG_CONTIGS genome + contig table, ARB_XG_ANNOTATION gene / exon tables with their indices, ARB_XG_TABLE the resident
 *   fragment table, ARB_XG_MISMAP_STATE what arb_filter_mismappers reads besides (candidate state and lists, fragment labels, k-mer index, splice sites).
 *   Sender: arb_exchange_header -> header words. Receiver: arb_exchange_prepare(header) sizes its buffers. Both: arb_exchange_buffers lists the same
 *   device buffers in the same order (the caller broadcasts each). Receiver: arb_exchange_commit. */
enum { ARB_XG_CONTIGS = 0, ARB_XG_ANNOTATION = 1, ARB_XG_TABLE = 2, ARB_XG_MISMAP_STATE = 3 };
int arb_exchange_header(arb_ctx* ctx, int group, uint64_t* header /* capacity 16 */, uint32_t* n_words);
int arb_exchange_prepare(arb_ctx* ctx, int group, const uint64_t* header, uint32_t n_words);
int arb_exchange_buffers(arb_ctx* ctx, int group, void** device_ptrs, uint64_t* bytes, uint32_t* n /* in: capacity (32 suffice), out: buffers */);
int arb_exchange_commit(arb_ctx* ctx, int group);
/* contig pairs (keys = lower contig << 16 | higher contig, ascending) and the part that owns each; fragments of other pairs emit no breakpoints in
 * arb_find_fusions. parts == 1 lifts the restriction. (arb_pipeline_work_partition computes a balanced assignment.) */
int arb_set_work_partition(arb_ctx* ctx, const uint32_t* keys, const uint8_t* owner, uint32_t n_keys, int part, int parts);
/* the part's candidate table packed into ONE device buffer (sizes = {candidates, list1, list2, listd entries}); after an all-gather of the buffers (padded
 * to `stride`) every part merges them into the table a single GPU would have built: candidates in first-insertion order (fusions.cpp:253-300) */
int arb_candidates_export(arb_ctx* ctx, void** device_blob, uint64_t* bytes, uint64_t sizes[4]);
int arb_candidates_import(arb_ctx* ctx, const void* all_blobs /* device */, uint64_t stride, const uint64_t* sizes /* 4 per part */, uint32_t n_parts);
/* canonical mate order (fusions.cpp:414-421) of the fragments other parts listed: arb_swaps_buffer = one byte per fragment on the device (1 = this part
 * exchanged MATE1/MATE2), combined by the caller with a MAX all-reduce in place; arb_swaps_apply performs the exchanges this part has not done */
int arb_swaps_buffer(arb_ctx* ctx, void** device_ptr, uint64_t* bytes);
int arb_swaps_apply(arb_ctx* ctx);
/* arb_filter_mismappers in two steps: _part re-aligns work items part, part + parts, ... and leaves one verdict byte per fragment on the device (combined by
 * the caller with a MAX all-reduce in place: filter_mismappers.cpp:232-244 only counts verdicts); _finish labels fragments and candidates */
int arb_filter_mismappers_part(arb_ctx* ctx, int32_t max_mate_gap, int part, int parts, void** device_verdicts, uint64_t* bytes);
int arb_filter_mismappers_finish(arb_ctx* ctx, uint64_t* n_realigned);

/* ---- device timing (CUDA events recorded on the context's stream around each stage) ---------------------------------- */
typedef struct arb_timings {
	float duplicates_ms;        /* duplicate marking (key build + hash group-by + mark) */
	float classify_ms;          /* the read-level cascade: both launches and the queue hand-over between them */
	float read_filters_ms;      /* whole arb_run_read_filters */
	float find_fusions_ms;      /* whole arb_find_fusions */
	uint64_t classify_algorithmic_bytes; /* SURVEY.md section 8(d) column budget of the cascade for the resident chunk (see cascade_algorithmic_bytes for what the launches actually saw) */
	uint64_t h2d_bytes;         /* bytes copied by the last arb_push_chunk */
	float h2d_ms;               /* duration of those copies */
	float merge_adjacent_ms, evalue_ms, kmer_index_ms, homologs_ms, mismappers_ms; /* candidate-level device stages */
	uint64_t mismapper_items;   /* (candidate, read) pairs re-aligned */
	uint64_t kmer_positions;    /* positions in the k-mer index */
	uint64_t mismapper_heavy_items; /* pairs that exhausted the one-thread budget and were re-aligned cooperatively */
	float mismappers_pass1_ms, mismappers_pass2_ms;
	uint64_t mismapper_tasks; uint32_t mismapper_rounds, mismapper_overflow, mismapper_table_slots; /* continuations re-aligned as tasks of their own, and the rounds that took */
	float cascade_head_ms, cascade_sequences_ms; /* the two launches of the read-level cascade (classify_ms spans both) */
	uint64_t cascade_queued;    /* fragments the sequence rules (mismatches, low entropy) looked at */
	uint64_t cascade_algorithmic_bytes[2]; /* SURVEY.md section 8(d) column budget of the two launches */
	float annotate_ms;          /* arb_annotate_pass1 + arb_annotate_pass2 (kernels, sorts and scans on the context's stream) */
	float in_vitro_ms;          /* arb_filter_in_vitro */
	float multimappers_ms;      /* arb_filter_multimappers */
	float order_ms;             /* arb_replay_insertion_order */
	float partners_ms;          /* arb_partner_counts */
	float rows_ms;              /* arb_format_discarded_rows */
	float bam_scan_ms;          /* arb_bam_scan, summed over the chunks of the last sample (copy + kernels + lists back) */
	float consensus_ms;         /* arb_build_consensus, summed over the batches of the last sample */
	float reserved_ms;
	uint64_t mismapper_algorithmic_bytes; /* SURVEY.md section 8(d) budget of pass 1 of the re-alignment: per searched sequence of length l, 3l/8 + 8(l-8) + 4*hits + l/2 */
	uint64_t mismapper_sequences, mismapper_hits; /* sequences searched by pass 1 (segment x gene x strand) and k-mer hits they visited */
} arb_timings;
int arb_get_timings(arb_ctx* ctx, arb_timings* out);
/* Device scratch memory is pooled per device and survives arb_ctx_destroy so that the next sample reuses it; this returns it to the driver
 * (no-op while a context on the current device still holds blocks). */
void arb_release_device_memory(void);
/* Large host columns are recycled the same way (first touch of fresh pages is what costs); this returns the free ones to the system. */
void arb_release_host_memory(void);

/* ---- whole-run driver ---------------------------------------------------------------------------------------
 * What the `arriba` executable does (source/arriba.cpp:79-631): reference + annotation loading, BAM ingest
 * (read_chimeric_alignments, source/read_chimeric_alignments.cpp:560), annotation (arriba.cpp:165-325), then the device
 * stages above. Host work is C++ on `threads` host threads; all device work goes through the entry points above. */
typedef struct arb_pipeline arb_pipeline;
typedef struct arb_run_options {
	const char* bam_file;            /* -x */
	const char* gtf_file;            /* -g */
	const char* assembly_file;       /* -a */
	const char* output_file;         /* -o (may be NULL until the writer stage is requested) */
	const char* discarded_output_file; /* -O or NULL */
	const char* interesting_contigs; /* -i or NULL for the default */
	const char* viral_contigs;       /* -v or NULL for the default */
	arb_params params;
	int32_t strandedness;            /* -s: 0 no, 1 yes, 2 reverse, 3 auto */
	uint32_t fragment_length;        /* -F 200 */
	int32_t threads;                 /* host threads */
	int32_t device;                  /* CUDA device ordinal */
	/* thresholds of the host-side event filters (defaults: source/options.cpp:71-107) */
	int32_t min_support;             /* -S 2 */
	uint32_t min_anchor_length;      /* -A 23 */
	uint32_t min_spliced_events;     /* -M 4 */
	float high_expression_quantile;  /* -Q 0.998 */
	float exonic_fraction;           /* -e 0.33 */
	float min_itd_allele_fraction;   /* -z 0.07 */
	uint32_t min_itd_support;        /* -Z 10 */
	int32_t print_extra_info_for_discarded_fusions; /* -X */
	int32_t echo_progress;           /* print the reference's progress lines to stdout while running */
	uint32_t top_viral_contigs;      /* -T 5 */
	float viral_contig_min_covered_fraction; /* -C 0.05 */
} arb_run_options;
void arb_default_run_options(arb_run_options* o);

enum { ARB_STEP_LOAD_REFERENCE = 0, ARB_STEP_INGEST = 1, ARB_STEP_ANNOTATE = 2, ARB_STEP_UPLOAD = 3, ARB_STEP_READ_FILTERS = 4,
       ARB_STEP_FRAGMENT_LENGTH = 5, ARB_STEP_FIND_FUSIONS = 6, ARB_STEP_COUNT = 7 };

typedef struct arb_run_stats {
	uint64_t n_fragments, n_records, mapped_reads, malformed;
	int32_t strandedness, max_mate_gap, fragment_length_ok;
	float mate_gap_mean, mate_gap_stddev, read_length_mean;
	double seconds[ARB_STEP_COUNT];      /* wall time per step */
	double t_inflate, t_parse, t_finalize; /* inside ARB_STEP_INGEST */
	uint64_t h2d_bytes;                  /* bytes copied host->device by ARB_STEP_UPLOAD */
	double event_seconds[32];            /* wall time per event-level stage (ARB_EV_*) */
	double output_seconds;               /* arb_pipeline_write_output */
	uint64_t n_candidates, n_unfiltered_candidates;
} arb_run_stats;

int arb_pipeline_create(arb_pipeline** out, const arb_run_options* options);
void arb_pipeline_destroy(arb_pipeline* p);
const char* arb_pipeline_error(arb_pipeline* p);   /* p may be NULL: error of arb_pipeline_create */
int arb_pipeline_step(arb_pipeline* p, int step);  /* steps must be run in order */
/* One sample on several GPUs (the device side: "one sample on several GPUs" above; arriba_b200/sharded.py is the launcher-side driver). The part that
 * ingests the BAM runs the pipeline as usual; it replicates its resident state to the other parts (arb_exchange_*), which only hold a context
 * (arb_pipeline_attach_device: the run's parameters, no host data). arb_pipeline_work_partition (after ARB_STEP_ANNOTATE) assigns the contig pairs to the
 * parts: keys ascending, owner[k] = part of keys[k]; pairs linked by duplicates stay together; heaviest first to the lightest part.
 * arb_pipeline_mismappers_begin runs the event chain up to, not including, filter_mismappers and sends the stage's inputs to the device (active = 0: the
 * stage is switched off); the launcher then calls arb_filter_mismappers_part / _finish on the contexts; arb_pipeline_mismappers_end takes the results back
 * and the chain resumes with arb_pipeline_events. */
int arb_pipeline_attach_device(arb_pipeline* p);
int arb_pipeline_work_partition(arb_pipeline* p, int parts, const uint32_t** keys, const uint8_t** owner, uint32_t* n_keys);
int arb_pipeline_mismappers_begin(arb_pipeline* p, int* active);
int arb_pipeline_mismappers_end(arb_pipeline* p);
int arb_pipeline_run(arb_pipeline* p);             /* all steps */
arb_ctx* arb_pipeline_ctx(arb_pipeline* p);        /* device context (valid after ARB_STEP_UPLOAD) */
int arb_pipeline_stats(arb_pipeline* p, arb_run_stats* out);
/* read-only view of the host fragment table (valid until the pipeline is destroyed); names: "<qname>,<HI>" concatenated */
int arb_pipeline_fragments(arb_pipeline* p, arb_soa_chunk* view, const char** names, const uint64_t** name_off /* n+1 */);
/* gene table after annotation (dummy genes included) and coverage windows of one contig */
int arb_pipeline_genes(arb_pipeline* p, arb_annotation* view);
int arb_pipeline_coverage(arb_pipeline* p, uint32_t contig, const uint16_t** coverage, const uint8_t** starts, const uint8_t** ends, uint64_t* n_windows);

/* event-level chain (source/arriba.cpp:420-545): runs the stages up to and including `last_stage` (ARB_EV_*) */
enum { ARB_EV_FETCH = 0, ARB_EV_MERGE_ADJACENT, ARB_EV_MULTIMAPPERS, ARB_EV_EVALUE, ARB_EV_NON_CODING_NEIGHBORS, ARB_EV_INTRAGENIC_EXONIC, ARB_EV_MIN_SUPPORT,
       ARB_EV_RELATIVE_SUPPORT, ARB_EV_ITD, ARB_EV_INTRONIC, ARB_EV_IN_VITRO, ARB_EV_SPLICED, ARB_EV_SELECT_BEST, ARB_EV_MARGINAL_READ_THROUGH, ARB_EV_MANY_SPLICED,
       ARB_EV_SHORT_ANCHOR, ARB_EV_END_TO_END, ARB_EV_NO_COVERAGE, ARB_EV_KMER_INDEX, ARB_EV_HOMOLOGS, ARB_EV_MISMAPPERS, ARB_EV_SELECT_BEST2, ARB_EV_ISOFORMS,
       ARB_EV_CONFIDENCE, ARB_EV_COUNT };
int arb_pipeline_events(arb_pipeline* p, int last_stage);
/* Replaces write_fusions_to_file (source/output_fusions.cpp:1043): writes output_file / discarded_output_file of the run options */
int arb_pipeline_write_output(arb_pipeline* p);
/* read-only view of the host candidate table: the arb_candidates pointers alias pipeline memory; `order` = the reference's
   iteration order (candidate ids), `confidence` and the current fragment labels complete the state */
int arb_pipeline_candidates(arb_pipeline* p, arb_candidates* view, const uint32_t** order, const uint8_t** confidence, const uint8_t** fragment_labels);

#ifdef __cplusplus
}
#endif
#endif
