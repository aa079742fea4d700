// engine.h -- device-resident state of one arriba-b200 context and the stage drivers.
#pragma once
#include "model.h"
#include "prims.h"
#include "read_filters.h"
#include "../../include/arriba_b200.h"
#include <time.h>
#include <vector>
#include <string>

namespace arb {

// CUDA-event stopwatch on the context's stream (wall clock in the hostsim build)
struct stage_timer {
#ifdef ARB_DEVICE_BUILD
	cudaEvent_t a, b; cudaStream_t s;
	explicit stage_timer(const exec_ctx& ex): s(ex.stream) { ARB_CUDA_CHECK(cudaEventCreate(&a)); ARB_CUDA_CHECK(cudaEventCreate(&b)); ARB_CUDA_CHECK(cudaEventRecord(a, s)); }
	float stop() { float ms = 0; ARB_CUDA_CHECK(cudaEventRecord(b, s)); ARB_CUDA_CHECK(cudaEventSynchronize(b)); ARB_CUDA_CHECK(cudaEventElapsedTime(&ms, a, b)); return ms; }
	~stage_timer() { cudaEventDestroy(a); cudaEventDestroy(b); }
#else
	double t0;
	static double now() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }
	explicit stage_timer(const exec_ctx&): t0(now()) {}
	float stop() { return (float) (now() - t0); }
#endif
};


struct frag_store {
	u32 n; u32 max_seq_len; bool canonical_seq_layout; u64 n_seq_bytes;
	dbuf<u8> n_aln, fflags, filter, early, aflags, seq, swapped;
	dbuf<u16> contig, cigar_cnt, seq_len, genes_cnt;
	dbuf<i32> start, end;
	dbuf<u32> cigar_off, seq_off, genes_off, cigar, genes;
	frag_store(): n(0), max_seq_len(0), canonical_seq_layout(false), n_seq_bytes(0) {}
	frag_view view() const {
		frag_view v;
		v.n = n; v.n_aln = n_aln.ptr(); v.fflags = fflags.ptr(); v.filter = filter.ptr();
		v.contig = contig.ptr(); v.start = start.ptr(); v.end = end.ptr(); v.aflags = aflags.ptr();
		v.cigar_off = cigar_off.ptr(); v.cigar_cnt = cigar_cnt.ptr(); v.seq_off = seq_off.ptr(); v.seq_len = seq_len.ptr();
		v.genes_off = genes_off.ptr(); v.genes_cnt = genes_cnt.ptr(); v.cigar = cigar.ptr(); v.seq = seq.ptr(); v.genes = genes.ptr();
		return v;
	}
};

struct annot_store {
	u32 n_genes, n_exons, n_contigs;
	dbuf<u16> gene_contig; dbuf<i32> gene_start, gene_end, gene_exonic_length; dbuf<u8> gene_strand, gene_flags;
	dbuf<u32> exon_gene; dbuf<i32> exon_start, exon_end, exon_cds_start, exon_cds_end, exon_next_start; dbuf<u8> exon_flags;
	dbuf<u32> exon_region_begin, exon_region_off, exon_region_items, gene_region_begin, gene_region_off, gene_region_items;
	dbuf<i32> exon_region_end, gene_region_end;
	dbuf<u8> contig_flags; dbuf<u64> contig_seq_off; dbuf<u32> contig_len; dbuf<char> assembly; dbuf<u32> assembly4; bool assembly4_ok;
	std::vector<u8> h_contig_flags; std::vector<u32> h_contig_len;
	// host mirrors needed by host-side steps
	std::vector<u16> h_gene_contig; std::vector<i32> h_gene_start, h_gene_end; std::vector<u8> h_gene_strand, h_gene_flags;
	u64 assembly_bytes, assembly4_words; u32 n_exon_regions, n_exon_items, n_gene_regions, n_gene_items; // exact sizes of the buffers above (exchange.cu)
	annot_store(): n_genes(0), n_exons(0), n_contigs(0), assembly4_ok(false), assembly_bytes(0), assembly4_words(0), n_exon_regions(0), n_exon_items(0), n_gene_regions(0), n_gene_items(0) {}
	annot_view view() const {
		annot_view v;
		v.n_genes = n_genes; v.gene_contig = gene_contig.ptr(); v.gene_start = gene_start.ptr(); v.gene_end = gene_end.ptr();
		v.gene_strand = gene_strand.ptr(); v.gene_exonic_length = gene_exonic_length.ptr(); v.gene_flags = gene_flags.ptr();
		v.n_exons = n_exons; v.exon_gene = exon_gene.ptr(); v.exon_start = exon_start.ptr(); v.exon_end = exon_end.ptr();
		v.exon_cds_start = exon_cds_start.ptr(); v.exon_cds_end = exon_cds_end.ptr(); v.exon_next_start = exon_next_start.ptr(); v.exon_flags = exon_flags.ptr();
		v.n_contigs = n_contigs;
		v.exon_region_begin = exon_region_begin.ptr(); v.exon_region_end = exon_region_end.ptr(); v.exon_region_off = exon_region_off.ptr(); v.exon_region_items = exon_region_items.ptr();
		v.gene_region_begin = gene_region_begin.ptr(); v.gene_region_end = gene_region_end.ptr(); v.gene_region_off = gene_region_off.ptr(); v.gene_region_items = gene_region_items.ptr();
		v.exon_grid = 0; v.exon_grid_begin = 0; v.gene_grid = 0; v.gene_grid_begin = 0;
		v.contig_flags = contig_flags.ptr(); v.contig_seq_off = contig_seq_off.ptr(); v.contig_len = contig_len.ptr(); v.assembly = assembly.ptr(); v.assembly4 = assembly4_ok ? assembly4.ptr() : 0;
		return v;
	}
};

struct cand_store {
	u32 n; u64 n_list1, n_list2, n_listd;
	dbuf<u32> gene1, gene2, split_reads1, split_reads2, discordant_mates, list1_off, list2_off, listd_off, list1, list2, listd;
	dbuf<u16> contig1, contig2; dbuf<i32> bp1, bp2, anchor1, anchor2; dbuf<u8> dir1, dir2, filter, bits, bits2; dbuf<float> evalue;
	dbuf<u32> first_frag; // fragment whose record created the candidate (merge key of the sharded run)
	cand_store(): n(0), n_list1(0), n_list2(0), n_listd(0) {}
};

struct exchange_buffer { void* p; u64 bytes; };

class engine {
public:
	scratch_set scratch; // scan / radix-sort scratch of this context (its device, its stream)
	exec_ctx ex;
	std::string last_error;
	arb_params params;
	frag_store frags;
	annot_store annot;
	cand_store cands;
	dbuf<u8> mismatch_table; u32 table_n, table_k;
	hash_index table;
	dbuf<u32> label_counts;
	bool has_contigs, has_annotation, filters_done;
	arb_timings timings;

	engine();
	~engine();
	void set_contigs(const arb_contigs& c);
	void set_annotation(const arb_annotation& a);
	void set_contig_flags(const u8* flags, u32 n);
	void set_params(const arb_params& p) { params = p; }
	void push_chunk(const arb_soa_chunk& c) { push_chunk_begin(c); push_chunk_end(c); }
	void push_chunk_begin(const arb_soa_chunk& c); // everything but the annotation columns (aflags, gene sets), asynchronously on the copy stream
	void push_chunk_end(const arb_soa_chunk& c);   // the annotation columns; returns when the whole table is resident
	// the fragment table built on the device from the ingest workers' pools (fragtable.cu): resident afterwards as after push_chunk_begin
	void build_fragment_table(const arb_ingest_pool* pools, u32 n_pools, arb_fragment_table_sizes& sizes); void get_fragment_table(const arb_fragment_columns& out);
	dbuf<char> ft_names, ft_out_names; dbuf<u32> ft_cigars, ft_frag_base; dbuf<u8> ft_seqs; dbuf<arb_pool_alignment> ft_alns; dbuf<arb_pool_fragment> ft_frags; dbuf<u64> ft_bases, ft_out_name_off;
	u64 ft_n_name_bytes; u32 tie_rounds;
	void table_resident(const exec_ctx& cx, u64 n_cigar, u64 n_seq_bytes); // bookkeeping once the ingest columns of frags.n fragments are on the device
	// device-side annotation of the resident chunk (annotate.cu): between the two passes the gene sets live in fixed rows + a pool
	u32 annotate_pass1(const u8* aflags, int strandedness); void get_dummy_genes(u16* contig, i32* start, i32* end); u64 annotate_pass2();
	void get_annotation_columns(u8* aflags, u32* genes_off, u16* genes_cnt, u32* genes);
	dbuf<u32> annot_rows, annot_pool, annot_ctl; dbuf<u16> annot_cnt; u32 annot_pool_cap, n_dummy; u64 n_gene_entries; dbuf<u16> dummy_contig; dbuf<i32> dummy_start, dummy_end;
	void finish_push(u64 n_gene_ids); u64 push_cigar_ops; dbuf<u64> chunk_stats;
	// one sample on several GPUs (exchange.cu): replicated state travels as groups of device buffers, the work of find_fusions / filter_mismappers is divided
	void exchange_header(int group, std::vector<u64>& header); void exchange_prepare(int group, const u64* header, u32 n_words);
	void exchange_buffers(int group, std::vector<exchange_buffer>& out); void exchange_commit(int group);
	void set_work_partition(const u32* keys, const u8* owner, u32 n_keys, int part, int parts); int work_part, work_parts; dbuf<u8> work_owned;
	void candidates_export(void** blob, u64* bytes, u64 sizes[4]); void candidates_import(const void* all_blobs, u64 stride, const u64* sizes, u32 n_parts); dbuf<char> cand_blob;
	void swaps_buffer(void** p, u64* bytes); void swaps_apply(); dbuf<u8> swap_union;
	void filter_mismappers_part(i32 max_mate_gap, int part, int parts, void** verdicts, u64* bytes); u64 filter_mismappers_finish(); dbuf<u8> mismap_verdicts; u64 mismap_items_total; float mismap_ms_part;
	u64 n_splice_sites;
	exec_ctx copy_ex; bool push_open; // copy stream: H2D of a chunk overlaps with host work (annotation) and with kernels on `ex`
	void run_read_filters();
	void get_fragment_filters(u8* filter_out, u8* early_out);
	void set_fragment_filters(const u8* filter);
	void get_filter_counts(u32* counts);
	void find_fusions(i32 max_mate_gap);
	void get_candidates(arb_candidates& out);
	void get_slot_swaps(u8* out);
	void set_candidate_state(const u8* filter, const u32* s1, const u32* s2, const u32* dm, const float* ev);
	void get_candidate_state(u8* filter, u32* s1, u32* s2, u32* dm, float* ev);
	void set_candidate_lists(const u32* l1o, const u32* l1, const u32* l2o, const u32* l2);
	u32 merge_adjacent(i32 max_distance);
	void get_merge_log(u32* triples, u32 n);
	void estimate_evalues(const arb_evalue_inputs& in);
	void filter_relative_support(float cutoff); void filter_multimappers(); u32 filter_simple(int stage, float exonic_fraction, int min_support); void evalue_tallies(u32* out); u32 select_best();
	void replay_insertion_order(const u32* phase_start, const u64* phase_buckets, u32 n_phases, u32* order_out, u32* rank_out); dbuf<u32> order_rank;
	void partner_counts(i32* count_out); dbuf<u32> order_seq;
	// BAM record boundaries and per-worker record lists of an inflated chunk (bamscan.cu)
	void bam_scan(const u8* chunk, u64 bytes, u64 first, i32 n_ref, u32 n_shards, u64* consumed, u32* n_records, u32* shard_begin, u32* record_offsets, u32* malformed); dbuf<u8> bam_buf;
	// rows of the discarded-fusions file (rows.cu)
	void set_row_texts(const arb_row_texts& t); void format_discarded_rows(const u8* confidence, u64* n_rows, u64* n_bytes); void get_row_text(char* out);
	dbuf<char> row_gene_name, row_gene_id, row_contig_name, row_filter_name, row_text; dbuf<u32> row_gene_name_off, row_gene_id_off, row_contig_name_off, row_filter_name_off; dbuf<i32> row_exon_prev, row_exon_next;
	u8 row_filters_by_name[ARB_N_FILTERS]; u32 row_max_itd_length; bool has_row_texts; u64 row_text_bytes; struct cand_state make_state_for_rows();
	// pileups and consensus sequences of the rows of fusions.tsv (consensus.cu)
	void build_consensus(const u32* rows, u32 n_rows, arb_consensus_info& info); void get_consensus(u32* seq_off, u32* pos_off, u32* clip_off, u8* verdict, u32* non_template, char* seq, i32* pos, char* clip);
	dbuf<u32> cons_seq_off, cons_pos_off, cons_clip_off, cons_non_template; dbuf<u8> cons_verdict; dbuf<char> cons_seq, cons_clip; dbuf<i32> cons_pos; u32 cons_rows; u64 cons_seq_bytes, cons_pos_count, cons_clip_bytes;
	dbuf<u32> merge_log; u32 merge_log_n;
	// filter_in_vitro on the device (events.cu): coverage windows of the sample, expression per gene
	void set_coverage(const u16* const* per_contig, const u64* n_windows, u32 n_contigs); void reads_by_gene(u32* out);
	void filter_in_vitro(const u32* reads, u32 n_genes, u32 threshold, const u64* pairs, u64 n_pairs); void spliced_support(const u32* reads, u32 n_genes, u32 threshold, u32* support_out);
	dbuf<u16> coverage_windows; dbuf<u64> coverage_off; dbuf<u32> coverage_n; u32 coverage_contigs;
	// k-mer index / re-alignment
	dbuf<i32> kmer_pos; dbuf<u32> kmer_bucket_off; u32 kmer_index_contigs; u64 kmer_indexed;
	dbuf<u32> kmer_block_first, kmer_block_base; u32 kmer_block_shift, kmer_blocks; struct kmer_index_view index_view(); // block table of the index (mismap_hd.h)
	u64 push_alignments, push_bases; u64 head_bytes, sequence_bytes; // column budgets of the two cascade launches for the resident chunk
	size_t cascade_smem_bytes; u32 cascade_resident_blocks; // launch shape of the sequence kernel on this context's device
	int device;
	bool mismap_group_pass; u32 mismap_group_lanes; int mismap_budget, mismap_spawn_budget, mismap_min_blocks; u32 mismap_lanes, mismap_task_lanes, mismap_table_slots, homolog_lanes; // work control of the re-alignment passes (mismap_hd.h, realign_ctl)
	dbuf<u32> splice_off; dbuf<i32> splice_sites; bool has_splice_sites;
	void set_splice_sites(const u32* off, const i32* sites);
	u64 build_kmer_index(const u32* contig, const i32* start, const i32* end, u32 n, u32 n_index_contigs);
	void kmer_index_digest(u64* kmers, u64* positions, u64* checksum, u32 n_contigs);
	void homolog_pairs(const u32* ga, const u32* gb, u32 n, u8* out);
	u64 filter_mismappers(i32 max_mate_gap);
	void set_candidates(const arb_candidates& c); void apply_slot_swaps(const u8* swapped); void get_first_fragments(u32* out);
	void probe_mismatch_counts(u32* out); // test hook (arb_selftest_mismatch_counts)
private:
	read_filter_params make_filter_params();
	unsigned long genome_size() const;
};

void default_params(arb_params& p);

} // namespace arb
