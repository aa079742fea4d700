// pipeline.h -- host-side orchestration of one arriba run: reference loading, BAM ingest, annotation, device stages
// (through the public C ABI only), event-level logic and output. Mirrors the call sequence of the reference's
// main (arriba.cpp:79-631).
#pragma once
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <thread>
#include <vector>
#include "refdata.h"
#include "ingest.h"
#include "events.h"
#include "../../../include/arriba_b200.h"

namespace arb { namespace host {

// ARB_TRACE=1: wall time of the parts of a stage, on stderr
struct stage_laps {
	const char* stage; bool on; double last;
	static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
	explicit stage_laps(const char* s): stage(s), on(getenv("ARB_TRACE") != NULL), last(now()) {}
	void lap(const char* what) { if (!on) return; const double t = now(); fprintf(stderr, "[laps] %-22s %-34s %8.1f ms\n", stage, what, (t - last) * 1e3); last = t; }
};

struct run_options { // options_t (options.hpp:25-69) restricted to what this implementation consumes
	std::string bam_file, gtf_file, assembly_file, output_file, discarded_output_file;
	std::string interesting_contigs, viral_contigs;
	arb_params params;
	int strandedness;          // 0 no, 1 yes, 2 reverse, 3 auto
	unsigned fragment_length;  // -F 200
	int threads;               // host threads for decode/annotation (the reference's -@ only affects BAM decoding)
	int device;
	bool print_extra_info_for_discarded_fusions; // -X
	int min_support; unsigned min_anchor_length, min_spliced_events, min_itd_support; float high_expression_quantile, exonic_fraction, min_itd_allele_fraction; bool echo_progress;
	unsigned top_viral_contigs; float viral_contig_min_covered_fraction; // -T 5, -C 0.05
	run_options();
};

struct pipeline {
	run_options opt; int threads;
	refdata ref; fragment_table frags; coverage_windows coverage; ingest_stats istats;
	arb_ctx* ctx;
	int strandedness; i32 max_mate_gap; float read_length_mean, mate_gap_mean, mate_gap_stddev; bool fragment_length_ok;
	std::vector<u8> labels, early;
	event_table ev;
	// ev.order (the reference's iteration order of its candidate map) is computed by fetch_candidates on the device
	void order_ready(); void replay_iteration_order();
	void say(const std::string& line); // appends to `log`, echoes with a time stamp when opt.echo_progress
	std::string log; // the reference's progress lines (arriba.cpp:61-66 style, without time stamps)
	double t_events[32], t_output;
	double t_reference, t_ingest, t_annotate, t_upload, t_read_filters, t_fragment_length, t_find_fusions;
	pipeline(): ctx(NULL), strandedness(0), max_mate_gap(0), read_length_mean(0), mate_gap_mean(0), mate_gap_stddev(0), fragment_length_ok(false), splice_sites_ready(false), events_done(-1),
	            upload_begun(false), t_mismappers_begin(0), frags_on_device(false), reference_on_device(false), coverage_on_device(false), row_texts_on_device(false), contigs_on_device(0) { for (int q = 0; q < 32; ++q) t_events[q] = 0; t_output = 0; t_reference = t_ingest = t_annotate = t_upload = t_read_filters = t_fragment_length = t_find_fusions = 0; }
	~pipeline();
	void load_reference();
	void ingest();
	void annotate();
	void upload();
	void upload_reference(); void send_annotation(); void begin_upload(); bool upload_begun; // ingest leaves the fragment table resident; the genome follows before annotation
	void read_filters();
	void fragment_length();
	void find_fusions();
	// event level (events.cpp); device stages go through the C ABI
	void fetch_candidates(); void push_candidate_state(); void pull_candidate_state(); void log_remaining(const char* what);
	void merge_adjacent(); void filter_multimappers(); void estimate_evalues(); void filter_relative_support();
	void filter_non_coding_neighbors(); void filter_intragenic_both_exonic(); void filter_min_support(); void recover_internal_tandem_duplication();
	void filter_both_intronic(); void filter_in_vitro(); void recover_both_spliced(); void select_best(); void filter_marginal_read_through();
	void recover_many_spliced(); void filter_short_anchor(); void filter_end_to_end(); void filter_no_coverage(); void recover_isoforms(); void assign_confidence();
	void write_output();
	void make_kmer_index(); void filter_homologs(); void filter_mismappers(); bool splice_sites_ready;
	void find_top_expressed_genes(std::vector<u32>& reads_by_gene, std::vector<u8>& present, unsigned int& threshold, float quantile);
	float intronic_fraction(u32 gene);
	void events_until(int last_stage); // runs the event-level chain up to and including `last_stage` (EV_* below)
	int events_done;
	void run_all();
	// one sample on several GPUs (shard.cpp; device side csrc/exchange.cu): contig pairs assigned to the parts, the re-alignment stage in two halves
	std::vector<u32> partition_keys; std::vector<u8> partition_owner; void work_partition(int parts);
	bool mismappers_begin(); void mismappers_end(); double t_mismappers_begin;
	void ensure_coverage_on_device(); void attach_device(); // a part that only works on replicated device state: a context with the run's parameters
	bool frags_on_device, reference_on_device, coverage_on_device, row_texts_on_device; u32 contigs_on_device;
	void say_read_filter_counts();
};

enum { EV_FETCH = 0, EV_MERGE_ADJACENT, EV_MULTIMAPPERS, EV_EVALUE, EV_NON_CODING_NEIGHBORS, EV_INTRAGENIC_EXONIC, EV_MIN_SUPPORT, EV_RELATIVE_SUPPORT,
       EV_ITD, EV_INTRONIC, EV_IN_VITRO, EV_SPLICED, EV_SELECT_BEST, EV_MARGINAL_READ_THROUGH, EV_MANY_SPLICED, EV_SHORT_ANCHOR, EV_END_TO_END, EV_NO_COVERAGE,
       EV_KMER_INDEX, EV_HOMOLOGS, EV_MISMAPPERS, EV_SELECT_BEST2, EV_ISOFORMS, EV_CONFIDENCE, EV_COUNT };

extern const char* const FILTER_NAMES[38];
int detect_strandedness(pipeline& p);
void annotate_fragments(pipeline& p);
void viral_contig_decisions(pipeline& p); // viral.cpp
bool estimate_fragment_length(pipeline& p, const u8* early, float& gap_mean, float& gap_stddev, float& read_length_mean);

}} // namespace
