// pipeline.cpp -- see pipeline.h.
#include "pipeline.h"
#include <chrono>
#include <ctime>
#include <iostream>
#include <sstream>
#include <stdexcept>
#include <algorithm>

namespace arb { namespace host {

static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

run_options::run_options(): interesting_contigs("1 2 3 4 5 6 7 8 9 10 11 12 13 14 15 16 17 18 19 20 21 22 X Y AC_* NC_*"), viral_contigs("AC_* NC_*"),
	strandedness(3), fragment_length(200), threads(1), device(0), print_extra_info_for_discarded_fusions(false), min_support(2), min_anchor_length(23), min_spliced_events(4), min_itd_support(10),
	high_expression_quantile(0.998f), exonic_fraction(0.33f), min_itd_allele_fraction(0.07f), echo_progress(false), top_viral_contigs(5), viral_contig_min_covered_fraction(0.05f) { arb_default_params(&params); }

void pipeline::say(const std::string& line) {
	log += line; log += "\n";
	if (getenv("ARB_TRACE")) { static double last = now_s(); const double t = now_s(); fprintf(stderr, "[trace] +%8.1f ms  %s\n", (t - last) * 1e3, line.c_str()); last = t; }
	if (opt.echo_progress) { time_t now = time(0); char buf[64]; strftime(buf, sizeof(buf), "[%Y-%m-%dT%X]", localtime(&now)); std::cout << buf << " " << line << std::endl; }
}

pipeline::~pipeline() { if (ctx) arb_ctx_destroy(ctx); }

static void check(arb_ctx* ctx, int rc, const char* what) { if (rc != 0) throw std::runtime_error(std::string(what) + ": " + arb_last_error(ctx)); }

void pipeline::load_reference() {
	const double t0 = now_s();
	threads = std::max(1, opt.threads);
	const bool filter_contigs = opt.params.filter_mask >> F_uninteresting_contigs & 1;
	if (!filter_contigs) opt.interesting_contigs = "*"; // arriba.cpp:92-93
	ref.load_assembly(opt.assembly_file, opt.interesting_contigs);
	ref.load_gtf(opt.gtf_file);
	ref.build_exon_index();
	ref.build_gene_index();
	ref.compute_exonic_lengths();
	ref.flatten();
	// the genome goes to the device with the reference (once per process in a deployment that runs sample after sample); a BAM header that names contigs the
	// assembly does not have makes begin_upload() send the grown contig table again
	ref.set_contig_flags(opt.interesting_contigs, opt.viral_contigs);
	ref.flatten();
	if (getenv("ARB_EARLY_REFERENCE") == NULL || atoi(getenv("ARB_EARLY_REFERENCE")) != 0) upload_reference();
	t_reference = now_s() - t0;
}

void pipeline::ingest() {
	const double t0 = now_s();
	ingest_options io; io.external_duplicate_marking = opt.params.external_duplicate_marking; io.max_itd_length = opt.params.max_itd_length;
	io.interesting_contigs = opt.interesting_contigs; io.viral_contigs = opt.viral_contigs; io.threads = threads;
	attach_device(); io.scan_ctx = ctx;
	read_chimeric_alignments(opt.bam_file, ref, io, frags, coverage, istats);
	std::ostringstream s; s << "Reading chimeric alignments from '" << opt.bam_file << "' (total=" << frags.n << ")";
	say(s.str());
	if (getenv("ARB_EARLY_UPLOAD") == NULL || atoi(getenv("ARB_EARLY_UPLOAD")) != 0) begin_upload();
	t_ingest = now_s() - t0;
}

void pipeline::annotate() {
	const double t0 = now_s();
	ref.set_contig_flags(opt.interesting_contigs, opt.viral_contigs);
	ref.flatten();
	u32 marked = 0;
	for (u32 i = 0; i + 1 < frags.n; ++i) { // count adjacent pairs like mark_multimappers' return value
		const u64 a0 = frags.name_off[i], a1 = frags.name_off[i + 1], a2 = frags.name_off[i + 2];
		u64 la = a1 - a0, lb = a2 - a1;
		while (la > 0 && frags.names[a0 + la - 1] != ',') --la;
		while (lb > 0 && frags.names[a1 + lb - 1] != ',') --lb;
		const u64 sa = la > 0 ? la - 1 : a1 - a0, sb = lb > 0 ? lb - 1 : a2 - a1;
		if (sa == sb && std::equal(frags.names.begin() + a0, frags.names.begin() + a0 + sa, frags.names.begin() + a1)) ++marked;
	}
	{ std::ostringstream s; s << "Marking multi-mapping alignments (marked=" << marked << ")"; say(s.str()); }
	strandedness = opt.strandedness;
	if (opt.strandedness == 3) {
		strandedness = detect_strandedness(*this);
		say(std::string("Detecting strandedness (") + (strandedness == 1 ? "yes" : strandedness == 2 ? "reverse" : "no") + ")");
	}
	if (!upload_begun) begin_upload(); // the passes run on the device over the resident columns
	annotate_fragments(*this);
	viral_contig_decisions(*this); // per-contig verdicts of the two viral heuristics; no-op without viral contigs
	t_annotate = now_s() - t0;
}

void pipeline::attach_device() {
	if (!ctx) { if (arb_ctx_create(&ctx, opt.device) != 0) throw std::runtime_error(arb_last_error(NULL)); }
	check(ctx, arb_set_params(ctx, &opt.params), "arb_set_params");
}

void pipeline::upload_reference() {
	attach_device();
	const u32 nc = (u32) ref.contig_ids.size();
	if (reference_on_device && contigs_on_device == nc) return;
	std::vector<const char*> seqs(nc, (const char*) NULL);
	for (u32 c = 0; c < nc; ++c) if (ref.has_sequence(c)) seqs[c] = ref.sequence(c);
	arb_contigs contigs = {nc, ref.contig_flags.data(), ref.seq_len.data(), seqs.data()};
	check(ctx, arb_set_contigs(ctx, &contigs), "arb_set_contigs");
	reference_on_device = true; contigs_on_device = nc;
}

// end of ingest: the genome follows the fragment table, which ingest left resident on the device (arb_build_fragment_table); the annotation columns
// follow in annotate()
void pipeline::begin_upload() {
	ref.set_contig_flags(opt.interesting_contigs, opt.viral_contigs); // the contig table is complete once the BAM header has been read
	ref.flatten();
	upload_reference();
	upload_begun = true;
}

// gene / exon tables and their region indices (after annotate(): with the dummy genes)
void pipeline::send_annotation() {
	arb_annotation a;
	const u32 nc = (u32) ref.contig_ids.size();
	a.n_genes = (u32) ref.genes.size(); a.gene_contig = ref.f_gene_contig.data(); a.gene_start = ref.f_gene_start.data(); a.gene_end = ref.f_gene_end.data();
	a.gene_strand = ref.f_gene_strand.data(); a.gene_exonic_length = ref.f_gene_exonic_length.data(); a.gene_flags = ref.f_gene_flags.data();
	a.n_exons = (u32) ref.exons.size(); a.exon_gene = ref.f_exon_gene.data(); a.exon_start = ref.f_exon_start.data(); a.exon_end = ref.f_exon_end.data();
	a.exon_cds_start = ref.f_exon_cds_start.data(); a.exon_cds_end = ref.f_exon_cds_end.data(); a.exon_next_start = ref.f_exon_next_start.data(); a.exon_flags = ref.f_exon_flags.data();
	a.n_contigs = nc;
	a.exon_region_begin = ref.exon_index.begin.data(); a.exon_region_end = ref.exon_index.end.data(); a.exon_region_off = ref.exon_index.off.data(); a.exon_region_items = ref.exon_index.items.data();
	a.gene_region_begin = ref.gene_index.begin.data(); a.gene_region_end = ref.gene_index.end.data(); a.gene_region_off = ref.gene_index.off.data(); a.gene_region_items = ref.gene_index.items.data();
	check(ctx, arb_set_annotation(ctx, &a), "arb_set_annotation");
}

void pipeline::upload() {
	const double t0 = now_s();
	upload_reference();
	// the contig flags with the per-sample verdicts on viral contigs (the annotation went to the device with annotate())
	check(ctx, arb_set_contig_flags(ctx, ref.contig_flags.data(), (u32) ref.contig_ids.size()), "arb_set_contig_flags");
	upload_begun = false;
	frags_on_device = true;
	t_upload = now_s() - t0;
}

void pipeline::read_filters() {
	const double t0 = now_s();
	check(ctx, arb_run_read_filters(ctx), "arb_run_read_filters");
	labels.resize(frags.n); early.resize(frags.n);
	check(ctx, arb_get_fragment_filters(ctx, labels.data(), early.data()), "arb_get_fragment_filters");
	say_read_filter_counts();
	t_read_filters = now_s() - t0;
}

void pipeline::say_read_filter_counts() {
	// `(remaining=N)` of every stage follows from the label histogram, because the first hit wins and the order is fixed (arriba.cpp:327-409)
	u64 counts[ARB_N_FILTERS]; for (int k = 0; k < ARB_N_FILTERS; ++k) counts[k] = 0;
	for (size_t i = 0; i < labels.size(); ++i) ++counts[labels[i] < ARB_N_FILTERS ? labels[i] : 0];
	static const int order[] = {F_duplicates, F_uninteresting_contigs, F_viral_contigs, F_top_expressed_viral_contigs, F_low_coverage_viral_contigs, F_read_through,
		F_inconsistently_clipped, F_homopolymer, F_small_insert_size, F_long_gap, F_same_gene, F_hairpin, F_mismatches};
	u64 remaining = frags.n;
	std::ostringstream s;
	// ITD-shaped fragments re-labelled by low_entropy keep their original stage unknown; the cumulative count is exact only when none were re-labelled
	for (size_t k = 0; k < sizeof(order) / sizeof(order[0]); ++k) if (opt.params.filter_mask >> order[k] & 1) { remaining -= counts[order[k]]; s << "Filtering " << FILTER_NAMES[order[k]] << " (remaining=" << remaining << ")\n"; }
	s << "Filtering reads with low entropy (remaining=" << counts[F_none] << ")";
	say(s.str());
}

void pipeline::fragment_length() {
	const double t0 = now_s();
	fragment_length_ok = estimate_fragment_length(*this, early.data(), mate_gap_mean, mate_gap_stddev, read_length_mean);
	if (fragment_length_ok) max_mate_gap = std::max(0, (int) (mate_gap_mean + 3 * mate_gap_stddev)); // arriba.cpp:357-363
	else { max_mate_gap = (i32) opt.fragment_length; read_length_mean = (float) opt.fragment_length; }
	t_fragment_length = now_s() - t0;
}

void pipeline::find_fusions() {
	const double t0 = now_s();
	check(ctx, arb_find_fusions(ctx, max_mate_gap), "arb_find_fusions");
	t_find_fusions = now_s() - t0;
}

void pipeline::events_until(int last) { // arriba.cpp:420-545, filters enabled by default
	const u64 m = opt.params.filter_mask;
	auto on = [&](int f) { return (m >> f) & 1; };
	for (int s = events_done + 1; s <= last && s < EV_COUNT; ++s) {
		const double t0 = now_s();
		switch (s) {
			case EV_FETCH: fetch_candidates(); break;
			case EV_MERGE_ADJACENT: if (on(F_merge_adjacent)) merge_adjacent(); break;
			case EV_MULTIMAPPERS: if (on(F_multimappers)) filter_multimappers(); break;
			case EV_EVALUE: estimate_evalues(); break;
			case EV_NON_CODING_NEIGHBORS: if (on(F_non_coding_neighbors)) filter_non_coding_neighbors(); break;
			case EV_INTRAGENIC_EXONIC: if (on(F_intragenic_exonic)) filter_intragenic_both_exonic(); break;
			case EV_MIN_SUPPORT: if (on(F_min_support)) filter_min_support(); break;
			case EV_RELATIVE_SUPPORT: if (on(F_relative_support)) filter_relative_support(); break;
			case EV_ITD: if (on(F_internal_tandem_duplication)) recover_internal_tandem_duplication(); break;
			case EV_INTRONIC: if (on(F_intronic)) filter_both_intronic(); break;
			case EV_IN_VITRO: if (on(F_in_vitro)) filter_in_vitro(); break;
			case EV_SPLICED: if (on(F_spliced)) recover_both_spliced(); break;
			case EV_SELECT_BEST: if (on(F_select_best)) select_best(); break;
			case EV_MARGINAL_READ_THROUGH: if (on(F_marginal_read_through)) filter_marginal_read_through(); break;
			case EV_MANY_SPLICED: if (on(F_many_spliced)) recover_many_spliced(); break;
			case EV_SHORT_ANCHOR: if (on(F_short_anchor)) filter_short_anchor(); break;
			case EV_END_TO_END: if (on(F_end_to_end)) filter_end_to_end(); break;
			case EV_NO_COVERAGE: if (on(F_no_coverage)) filter_no_coverage(); break;
			case EV_KMER_INDEX: if (on(F_homologs) || on(F_mismappers)) make_kmer_index(); break;
			case EV_HOMOLOGS: if (on(F_homologs)) filter_homologs(); break;
			case EV_MISMAPPERS: if (on(F_mismappers)) filter_mismappers(); break;
			case EV_SELECT_BEST2: if (on(F_many_spliced) && on(F_select_best)) select_best(); break; // arriba.cpp:573-579
			case EV_ISOFORMS: if (on(F_isoforms)) recover_isoforms(); break;
			case EV_CONFIDENCE: assign_confidence(); break;
		}
		t_events[s] = now_s() - t0;
		events_done = s;
	}
}

void pipeline::run_all() { load_reference(); ingest(); annotate(); upload(); read_filters(); fragment_length(); find_fusions(); events_until(EV_COUNT - 1); write_output(); }

}} // namespace
