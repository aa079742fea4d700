// engine.cu -- stage drivers: uploads, duplicate marking, the fused read-level cascade.
#include <cstdlib>
#include <algorithm>
#include "engine.h"
#include "mismatch_table.h"

namespace arb {

void default_params(arb_params& p) { // options.cpp:71-107
	p.filter_mask = 0;
	for (u32 f = 1; f < F_COUNT; ++f) p.filter_mask |= (u64) 1 << f;
	p.homopolymer_length = 6; p.min_read_through_distance = 10000; p.max_kmer_content = 0.6f; p.max_itd_length = 100;
	p.external_duplicate_marking = 0; p.mismatch_pvalue_cutoff = 0.01f; p.subsampling_threshold = 300; p.evalue_cutoff = 0.3f;
	p.max_mismapper_fraction = 0.8f; p.max_homolog_identity = 0.3f;
}

engine::engine(): ft_n_name_bytes(0), tie_rounds(0), row_max_itd_length(0), has_row_texts(false), row_text_bytes(0), kmer_block_shift(0), kmer_blocks(0), coverage_contigs(0), work_part(0), work_parts(1), mismap_items_total(0), mismap_ms_part(0), n_splice_sites(0), annot_pool_cap(0), n_dummy(0), n_gene_entries(0), push_cigar_ops(0), cascade_smem_bytes(0), cascade_resident_blocks(0), device(0), table_n(0), table_k(0), has_contigs(false), has_annotation(false), filters_done(false), merge_log_n(0), kmer_index_contigs(0), kmer_indexed(0), has_splice_sites(false) {
	default_params(params);
	memset(&timings, 0, sizeof(timings));
	cons_rows = 0; cons_seq_bytes = cons_pos_count = cons_clip_bytes = 0;
	// tuning hooks of the re-alignment passes (mismap_hd.h): ARB_MISMAP_BUDGET (0 = thread-per-item only), ARB_MISMAP_LANES, ARB_MISMAP_SPAWN (0 = no task rounds), ARB_MISMAP_TASK_LANES
	mismap_group_pass = true; if (const char* s = getenv("ARB_MISMAP_GROUP")) mismap_group_pass = atoi(s) != 0;
	mismap_group_lanes = 16; if (const char* s = getenv("ARB_MISMAP_GROUP_LANES")) mismap_group_lanes = (u32) atoi(s);
	mismap_budget = 4096; mismap_lanes = 1024; mismap_spawn_budget = 0; mismap_task_lanes = 32;
	if (const char* s = getenv("ARB_MISMAP_BUDGET")) mismap_budget = atoi(s);
	if (const char* s = getenv("ARB_MISMAP_LANES")) mismap_lanes = (u32) std::max(1, atoi(s));
	if (const char* s = getenv("ARB_MISMAP_SPAWN")) mismap_spawn_budget = atoi(s);
	homolog_lanes = 32; if (const char* s = getenv("ARB_HOMOLOG_LANES")) homolog_lanes = (u32) std::max(1, atoi(s)); // threads per gene pair in filter_homologs' identity test (1 = one thread per pair)
	mismap_table_slots = 4096; if (const char* s = getenv("ARB_MISMAP_TABLE")) mismap_table_slots = (u32) std::max(1, atoi(s)); // continuation registry: slots provisioned per cooperative item (the table is shared, 2^20..2^25 slots)
	mismap_min_blocks = 4; if (const char* s = getenv("ARB_MISMAP_OCC")) mismap_min_blocks = atoi(s); // resident 256-thread blocks per SM the re-alignment kernels are compiled for
	if (const char* s = getenv("ARB_MISMAP_TASK_LANES")) mismap_task_lanes = (u32) std::max(1, atoi(s));
	ex.scratch = &scratch;
#ifdef ARB_DEVICE_BUILD
	ARB_CUDA_CHECK(cudaStreamCreateWithFlags(&ex.stream, cudaStreamNonBlocking));
	ARB_CUDA_CHECK(cudaStreamCreateWithFlags(&copy_ex.stream, cudaStreamNonBlocking));
#endif
	copy_ex.scratch = &scratch; push_open = false;
}

engine::~engine() { // arb_ctx_destroy has made the context's device current; buffers go back to that device's pool after the stream has drained
#ifdef ARB_DEVICE_BUILD
	if (copy_ex.stream) { cudaStreamSynchronize(copy_ex.stream); cudaStreamDestroy(copy_ex.stream); copy_ex.stream = 0; }
	if (ex.stream) { cudaStreamSynchronize(ex.stream); cudaStreamDestroy(ex.stream); ex.stream = 0; }
#endif
}

// reference bases as nt16 codes, eight per word: the mismatch rule compares eight read bases per XOR (read_filters.h)
struct pack_assembly_fn {
	const char* bases; u32 length; u32* packed; u32* exotic; // one contig; bases and packed start at the contig's (64-base aligned) offset
	ARB_HD void operator()(u32 w) const {
		u32 word = 0;
		for (u32 b = 0; b < 8 && w * 8 + b < length; ++b) {
			const u32 code = nt16_of_char(bases[w * 8 + b]);
			if (code > 15) { *exotic = 1; continue; }
			word |= code << (28 - 4 * b);
		}
		packed[w] = word;
	}
};

void engine::set_contigs(const arb_contigs& c) {
	annot.n_contigs = c.n_contigs;
	annot.h_contig_flags.assign(c.flags, c.flags + c.n_contigs);
	annot.h_contig_len.assign(c.length, c.length + c.n_contigs);
	std::vector<u64> off(c.n_contigs);
	u64 total = 0;
	for (u32 k = 0; k < c.n_contigs; ++k) {
		const bool loaded = c.sequence && c.sequence[k] && c.length[k] > 0;
		off[k] = loaded ? total : ~(u64) 0;
		if (!loaded) annot.h_contig_len[k] = 0;
		if (loaded) total += ((u64) c.length[k] + 63) & ~(u64) 63;
	}
	annot.assembly.ensure(total + 64); annot.assembly_bytes = total;
	for (u32 k = 0; k < c.n_contigs; ++k) {
		if (off[k] == ~(u64) 0) continue;
#ifdef ARB_DEVICE_BUILD
		ARB_CUDA_CHECK(cudaMemcpyAsync(annot.assembly.ptr() + off[k], c.sequence[k], c.length[k], cudaMemcpyHostToDevice, ex.stream));
#else
		memcpy(annot.assembly.ptr() + off[k], c.sequence[k], c.length[k]);
#endif
	}
	for (u32 k = 0; k < c.n_contigs; ++k) if (off[k] == ~(u64) 0) off[k] = 0; // contig_len == 0 guards every access
	annot.contig_flags.upload(ex, annot.h_contig_flags.data(), c.n_contigs);
	annot.contig_len.upload(ex, annot.h_contig_len.data(), c.n_contigs);
	annot.contig_seq_off.upload(ex, off.data(), c.n_contigs);
	{
		const u64 n_words = total / 8 + 9; // windows read one word past the last base
		annot.assembly4.ensure(n_words); annot.assembly4.zero(ex, n_words); annot.assembly4_words = n_words;
		dbuf<u32> exotic(1); exotic.zero(ex, 1);
		for (u32 k = 0; k < c.n_contigs; ++k) {
			if (annot.h_contig_len[k] == 0) continue;
			pack_assembly_fn pf = {annot.assembly.ptr() + off[k], annot.h_contig_len[k], annot.assembly4.ptr() + off[k] / 8, exotic.ptr()};
			for_each(ex, (annot.h_contig_len[k] + 7) / 8, pf);
		}
		u32 flag = 0; exotic.download(ex, &flag, 1);
		annot.assembly4_ok = flag == 0;
	}
	ex.sync();
	has_contigs = true;
	table_n = 0; // mismatch table depends on the genome size
}

void engine::set_contig_flags(const u8* flags, u32 n) { // per-sample flags (interesting / viral patterns, verdicts of the viral heuristics) without re-sending the genome
	if (!has_contigs || n != annot.n_contigs) throw arb_error("arb_set_contig_flags: contig table not set or of a different size");
	bool interesting_changed = false;
	for (u32 k = 0; k < n; ++k) if ((flags[k] ^ annot.h_contig_flags[k]) & CF_INTERESTING) interesting_changed = true;
	annot.h_contig_flags.assign(flags, flags + n);
	annot.contig_flags.upload(ex, annot.h_contig_flags.data(), n);
	ex.sync();
	if (interesting_changed) table_n = 0; // the mismatch table depends on the genome size (filter_mismatches.cpp:105-108)
}

void engine::set_annotation(const arb_annotation& a) {
	if (has_contigs && a.n_contigs != annot.n_contigs) throw arb_error("annotation and contig table disagree on the number of contigs");
	annot.n_genes = a.n_genes; annot.n_exons = a.n_exons; annot.n_contigs = a.n_contigs;
	annot.gene_contig.upload(ex, a.gene_contig, a.n_genes); annot.gene_start.upload(ex, a.gene_start, a.n_genes); annot.gene_end.upload(ex, a.gene_end, a.n_genes);
	annot.gene_strand.upload(ex, a.gene_strand, a.n_genes); annot.gene_exonic_length.upload(ex, a.gene_exonic_length, a.n_genes); annot.gene_flags.upload(ex, a.gene_flags, a.n_genes);
	annot.exon_gene.upload(ex, a.exon_gene, a.n_exons); annot.exon_start.upload(ex, a.exon_start, a.n_exons); annot.exon_end.upload(ex, a.exon_end, a.n_exons);
	annot.exon_cds_start.upload(ex, a.exon_cds_start, a.n_exons); annot.exon_cds_end.upload(ex, a.exon_cds_end, a.n_exons);
	annot.exon_next_start.upload(ex, a.exon_next_start, a.n_exons); annot.exon_flags.upload(ex, a.exon_flags, a.n_exons);
	const u32 ner = a.exon_region_begin[a.n_contigs], ngr = a.gene_region_begin[a.n_contigs];
	annot.n_exon_regions = ner; annot.n_gene_regions = ngr; annot.n_exon_items = a.exon_region_off[ner]; annot.n_gene_items = a.gene_region_off[ngr];
	annot.exon_region_begin.upload(ex, a.exon_region_begin, a.n_contigs + 1); annot.exon_region_end.upload(ex, a.exon_region_end, ner);
	annot.exon_region_off.upload(ex, a.exon_region_off, ner + 1); annot.exon_region_items.upload(ex, a.exon_region_items, a.exon_region_off[ner]);
	annot.gene_region_begin.upload(ex, a.gene_region_begin, a.n_contigs + 1); annot.gene_region_end.upload(ex, a.gene_region_end, ngr);
	annot.gene_region_off.upload(ex, a.gene_region_off, ngr + 1); annot.gene_region_items.upload(ex, a.gene_region_items, a.gene_region_off[ngr]);
	annot.h_gene_contig.assign(a.gene_contig, a.gene_contig + a.n_genes); annot.h_gene_start.assign(a.gene_start, a.gene_start + a.n_genes);
	annot.h_gene_end.assign(a.gene_end, a.gene_end + a.n_genes); annot.h_gene_strand.assign(a.gene_strand, a.gene_strand + a.n_genes);
	annot.h_gene_flags.assign(a.gene_flags, a.gene_flags + a.n_genes);
	ex.sync();
	has_annotation = true;
}

// The fragment table goes to the device in two parts. Everything ingest produces is final when ingest ends and is copied first, asynchronously on the
// copy stream (the caller's columns are page-locked when they were built in blocks of the host pool, arb_host_alloc) -- the caller annotates meanwhile;
// the annotation columns (alignment flags with the exonic / strand bits, gene sets) follow, and push_chunk_end returns when the table is resident.
struct chunk_stats_fn { // out: [0] longest sequence, [1] bases, [2] alignments, [3] breaks of the canonical pool layout
	frag_view f; unsigned long long* out;
	ARB_HD static void add(unsigned long long* p, unsigned long long v) {
#ifdef __CUDA_ARCH__
		atomicAdd(p, v);
#else
		*p += v;
#endif
	}
	ARB_HD static void take_max(unsigned long long* p, unsigned long long v) {
#ifdef __CUDA_ARCH__
		atomicMax(p, v);
#else
		if (v > *p) *p = v;
#endif
	}
	ARB_HD void operator()(u32 i) const {
		const u32 a0 = f.idx(i, 0), a1 = f.idx(i, 1);
		const u32 l0 = f.seq_len[a0], l1 = f.seq_len[a1];
		const u32 u0 = ((l0 + 1) / 2 + 15) / 16, u1 = ((l1 + 1) / 2 + 15) / 16;
		u32 breaks = 0;
		if (f.seq_off[a1] != f.seq_off[a0] + u0) ++breaks;
		if (i + 1 < f.n) { if (f.seq_off[f.idx(i + 1, 0)] != f.seq_off[a1] + u1) ++breaks; }
#ifdef __CUDA_ARCH__
		// one atomic per warp and statistic
		const unsigned active = __activemask();
		u32 mx = l0 > l1 ? l0 : l1, bases = l0 + l1, alns = f.n_aln[i];
		for (int d = 16; d; d >>= 1) { const u32 m2 = __shfl_xor_sync(active, mx, d), b2 = __shfl_xor_sync(active, bases, d), a2 = __shfl_xor_sync(active, alns, d), k2 = __shfl_xor_sync(active, breaks, d); mx = m2 > mx ? m2 : mx; bases += b2; alns += a2; breaks += k2; }
		if (active == 0xFFFFFFFFu) { if ((threadIdx.x & 31u) == 0) { take_max(out, mx); add(out + 1, bases); add(out + 2, alns); if (breaks) add(out + 3, breaks); } return; }
		mx = l0 > l1 ? l0 : l1; bases = l0 + l1; alns = f.n_aln[i]; breaks = (f.seq_off[a1] != f.seq_off[a0] + u0) + ((i + 1 < f.n) && f.seq_off[f.idx(i + 1, 0)] != f.seq_off[a1] + u1);
#else
		const u32 mx = l0 > l1 ? l0 : l1, bases = l0 + l1, alns = f.n_aln[i];
#endif
		take_max(out, mx); add(out + 1, bases); add(out + 2, alns); if (breaks) add(out + 3, breaks);
	}
};

void engine::push_chunk_begin(const arb_soa_chunk& c) {
	const u32 n = c.n_fragments;
	ex.sync(); // kernels of the previous sample may still read the buffers that are about to be overwritten
	frags.n = n;
	const exec_ctx& cx = copy_ex;
	stage_timer t_h2d(cx);
	frags.n_aln.upload(cx, c.n_aln, n); frags.fflags.upload(cx, c.fflags, n); frags.filter.upload(cx, c.filter, n);
	frags.contig.upload(cx, c.contig, 3 * (size_t) n); frags.start.upload(cx, c.start, 3 * (size_t) n); frags.end.upload(cx, c.end, 3 * (size_t) n);
	frags.cigar_off.upload(cx, c.cigar_off, 3 * (size_t) n); frags.cigar_cnt.upload(cx, c.cigar_cnt, 3 * (size_t) n);
	frags.seq_off.upload(cx, c.seq_off, 2 * (size_t) n); frags.seq_len.upload(cx, c.seq_len, 2 * (size_t) n);
	frags.cigar.upload(cx, c.cigar, c.n_cigar); frags.seq.upload(cx, c.seq, c.n_seq_bytes);
	table_resident(cx, c.n_cigar, c.n_seq_bytes);
	timings.h2d_ms = t_h2d.stop(); // waits for part one: the caller's annotation takes far longer than the copy, and the timing stays a pure copy time
	timings.h2d_bytes = (u64) n * 3 + (u64) n * 3 * (2 + 4 + 4 + 4 + 2) + (u64) n * 2 * (4 + 2) + c.n_cigar * 4 + c.n_seq_bytes;
}

void engine::table_resident(const exec_ctx& cx, u64 n_cigar, u64 n_seq_bytes) {
	const u32 n = frags.n;
	frags.early.ensure(n); frags.swapped.ensure(n); frags.swapped.zero(cx, n);
	// statistics of the chunk, taken on the device behind the copies (a pass over four columns: serial on the host it cost a tenth of a second per 10 M
	// fragments): longest sequence, bases, alignments, and whether the sequence pool has the canonical layout (what ingest writes: sequences in fragment
	// order, slot 0 then slot 1, back to back in 16-byte units -- the sequence kernel then stages a tile of fragments with one bulk copy)
	chunk_stats.ensure(8); chunk_stats.zero(cx, 8);
	chunk_stats_fn cs = {frags.view(), (unsigned long long*) chunk_stats.ptr()};
	for_each(cx, n, cs);
	u64 st[4] = {0, 0, 0, 0};
	chunk_stats.download(cx, st, 4);
	frags.max_seq_len = (u32) st[0];
	frags.n_seq_bytes = n_seq_bytes;
	frags.canonical_seq_layout = n > 0 && n_seq_bytes % 16 == 0 && st[3] == 0;
	push_alignments = st[2]; push_bases = st[1]; push_cigar_ops = n_cigar;
	push_open = true;
	filters_done = false;
	cands.n = 0;
}

void engine::push_chunk_end(const arb_soa_chunk& c) {
	if (!push_open || c.n_fragments != frags.n) throw arb_error("arb_push_chunk_end without a matching arb_push_chunk_begin");
	const u32 n = c.n_fragments;
	const exec_ctx& cx = copy_ex;
	stage_timer t_h2d(cx);
	frags.aflags.upload(cx, c.aflags, 3 * (size_t) n);
	frags.genes_off.upload(cx, c.genes_off, 3 * (size_t) n); frags.genes_cnt.upload(cx, c.genes_cnt, 3 * (size_t) n); frags.genes.upload(cx, c.genes, c.n_genes);
	timings.h2d_ms += t_h2d.stop();
	timings.h2d_bytes += (u64) n * 3 * (1 + 4 + 2) + c.n_genes * 4;
	cx.sync();
	finish_push(c.n_genes);
}

// the resident table is complete: column budget of the cascade launches for it
void engine::finish_push(u64 n_gene_ids) {
	const u32 n = frags.n;
	// Column budget of SURVEY.md section 8(d): every column read once at its compact width -- 11 B per alignment {contig u16, start, end, flags u8}, CIGAR ops and
	// gene ids with a 4-byte offset per alignment, 6 B per fragment {rank, flags, label}; sequences at 3 bit/base, gathered reference bases at 2 bit/base.
	const u64 n_alignments = push_alignments, bases = push_bases;
	head_bytes = n_alignments * 11 + (push_cigar_ops + n_alignments) * 4 + (n_gene_ids + n_alignments) * 4 + (u64) n * 6;
	sequence_bytes = bases * 3 / 8 + bases * 2 / 8 + (push_cigar_ops + n_alignments) * 4 + n_alignments * 11 + (u64) n * 2;
	timings.classify_algorithmic_bytes = head_bytes + sequence_bytes;
	push_open = false;
#ifdef ARB_DEVICE_BUILD
	{ // realign() (mismap_hd.h) recurses once per continuation, each at least 8 read bases further on, reads of 300 bases and more are not re-aligned: frames of < 512 B
		const size_t levels = std::min<size_t>(frags.max_seq_len, 300) / 8 + 4, wanted = 1024 + 512 * levels;
		size_t have = 0;
		if (cudaDeviceGetLimit(&have, cudaLimitStackSize) == cudaSuccess && have < wanted) ARB_CUDA_CHECK(cudaDeviceSetLimit(cudaLimitStackSize, wanted));
	}
#endif
}

unsigned long engine::genome_size() const { // filter_mismatches.cpp:105-108
	unsigned long g = 0;
	for (u32 k = 0; k < annot.n_contigs; ++k) if (annot.h_contig_flags[k] & CF_INTERESTING) g += annot.h_contig_len[k];
	return g;
}

read_filter_params engine::make_filter_params() {
	// decision table large enough for every (aligned bases, mismatches) the resident fragments can produce
	const u32 need_n = frags.max_seq_len + 2, need_k = frags.max_seq_len + 70;
	if (table_n < need_n || table_k < need_k) {
		table_n = need_n; table_k = need_k;
		std::vector<u8> t = build_mismatch_table(table_n, table_k, 0.01f /* arriba.cpp:403 */, genome_size(), params.mismatch_pvalue_cutoff);
		mismatch_table.upload(ex, t.data(), t.size());
		ex.sync();
	}
	read_filter_params p;
	p.stage_mask = (u32) params.filter_mask; p.stage_mask_hi = (u32) (params.filter_mask >> 32);
	p.homopolymer_length = params.homopolymer_length; p.min_read_through_distance = params.min_read_through_distance;
	p.max_overhang = 5; p.max_kmer_content = params.max_kmer_content; p.max_itd_length = params.max_itd_length;
	p.external_duplicate_marking = params.external_duplicate_marking;
	p.mismatch_table = mismatch_table.ptr(); p.table_n = table_n; p.table_k = table_k;
	return p;
}

// ------------------------------------------------------------------------------------------- duplicate marking
struct dup_key_fn { // pass 1: compact 12-byte keys, coalesced
	frag_view f; u64* k0; u32* k1; u8* participate;
	ARB_HD void operator()(u32 i) const {
		const dup_key k = duplicate_key(f, i);
		k0[i] = (u64) (u32) k.p1 | (u64) (u32) k.p2 << 32; k1[i] = (u32) k.c1 | (u32) k.c2 << 16;
		participate[i] = f.filter[i] == F_none;
	}
};
struct dup_key_ops {
	const u64* k0; const u32* k1;
	ARB_HD u64 hash(u32 i) const { dup_key k; k.p1 = (i32) (u32) k0[i]; k.p2 = (i32) (u32) (k0[i] >> 32); k.c1 = (u16) k1[i]; k.c2 = (u16) (k1[i] >> 16); return dup_hash(k); }
	ARB_HD bool equal(u32 a, u32 b) const { return k0[a] == k0[b] && k1[a] == k1[b]; }
};
struct dup_mark_fn {
	const u32* first; const u8* participate; u8* filter;
	ARB_HD void operator()(u32 i) const { if (participate[i] && first[i] != i) filter[i] = F_duplicates; }
};
struct dup_external_fn {
	frag_view f;
	ARB_HD void operator()(u32 i) const { if (f.filter[i] == F_none && (f.fflags[i] & FF_DUPLICATE)) f.filter[i] = F_duplicates; }
};

// ------------------------------------------------------------------------------------------- the cascade, two kernels
struct cascade_head_fn {
	read_filter_params p; frag_view f; annot_view an; u8* early; u8* needs_sequences; u32* n_queued;
	ARB_HD void operator()(u32 i) const {
		u8 e; bool more;
		const u8 label = classify_head(p, f, an, i, e, more);
		f.filter[i] = label; early[i] = e;
		needs_sequences[i] = more;
		if (more) append_slot(n_queued); // one atomic per warp: how many fragments the sequence rules will look at
	}
};
struct cascade_sequences_fn { // one thread per fragment: host build only (the device runs k_cascade_sequences)
	read_filter_params p; frag_view f; annot_view an; const u8* needs_sequences;
	ARB_HD void operator()(u32 i, u32* scratch, u32 stride) const { if (needs_sequences[i]) f.filter[i] = classify_sequences(p, f, an, i, scratch, stride); }
};

#ifdef ARB_DEVICE_BUILD
// The sequence rules (mismatches, low entropy): CASCADE_LANES lanes per fragment, a warp takes four consecutive fragments at a time.
//  * the read sequences of a warp's fragments are one contiguous stretch of the sequence pool (fragments lie in name order, slots 0 and 1 back to back): ONE bulk
//    copy (cp.async.bulk, completion on the warp's mbarrier) brings it to shared memory while the lanes fetch the fragments' columns; a chunk whose pool is
//    laid out differently (arb_push_chunk accepts any offsets) is read in place;
//  * the lanes of a group take the 8-base words of a read in turn: reference words are read 32 bytes per group and load, 3-mers are counted with
//    shared-memory atomics into the group's 64 counters (read_filters.h, classify_sequences_group).
// Persistent grid: the warps stride over the tiles.
static const u32 CASCADE_LANES = 8, CASCADE_THREADS = 256, CASCADE_GROUPS = CASCADE_THREADS / CASCADE_LANES, CASCADE_GROUPS_PER_WARP = 32 / CASCADE_LANES;
struct cascade_tile_params { u32 group_words /* 64 counters + dense codes + predecessor masks, per group */; u32 seq_capacity_units /* 16-byte units of staging room per warp, 0 = read in place */; u32 n_seq_units /* size of the sequence pool */; };

__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64* bar, u32 count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(u64* bar, u32 bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory"); }
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, u32 bytes, u64* bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64* bar, u32 parity) {
	asm volatile("{\n.reg .pred p;\nWAIT_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}

__global__ void __launch_bounds__(CASCADE_THREADS) k_cascade_sequences(read_filter_params p, frag_view f, annot_view an, const u8* __restrict__ needs_sequences, cascade_tile_params tp) {
	// Every WARP works on its own: a tile is the CASCADE_GROUPS_PER_WARP consecutive fragments of one warp, staged by the warp's own bulk copy on the warp's own
	// mbarrier -- no block-wide barrier, so a fragment that takes long (many alignment blocks, a long read) holds up three neighbours, not a block.
	extern __shared__ __align__(128) u8 smem[];
	const u32 warp = threadIdx.x / 32, lane32 = threadIdx.x & 31u, group_in_warp = lane32 / CASCADE_LANES;
	const u32 warp_seq_bytes = tp.seq_capacity_units * 16; // staging room of one warp
	u8* const staged = smem + (size_t) warp * warp_seq_bytes;
	u32* const counters = (u32*) (smem + (size_t) (CASCADE_THREADS / 32) * warp_seq_bytes) + (size_t) (threadIdx.x / CASCADE_LANES) * tp.group_words;
	__shared__ __align__(8) u64 bars[CASCADE_THREADS / 32];
	u64* const bar = &bars[warp];
	lane_group g; g.lane = threadIdx.x % CASCADE_LANES; g.lanes = CASCADE_LANES; g.mask = ((1u << CASCADE_LANES) - 1u) << (group_in_warp * CASCADE_LANES);
	if (lane32 == 0) { mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
	__syncwarp();
	u32 parity = 0;
	const u32 n_tiles = (f.n + CASCADE_GROUPS_PER_WARP - 1) / CASCADE_GROUPS_PER_WARP;
	const u32 n_warps = gridDim.x * (CASCADE_THREADS / 32);
	for (u32 tile = blockIdx.x * (CASCADE_THREADS / 32) + warp; tile < n_tiles; tile += n_warps) {
		const u32 first = tile * CASCADE_GROUPS_PER_WARP, end = hd_min(first + CASCADE_GROUPS_PER_WARP, f.n);
		const u32 i = first + group_in_warp;
		const bool mine = i < end && needs_sequences[i];
		if (!__any_sync(0xFFFFFFFFu, mine)) continue;
		u32 lo = 0, units = 0;
		if (tp.seq_capacity_units) { // canonical pool: the tile's sequences end where the next fragment's begin
			if (lane32 == 0) {
				lo = f.seq_off[first];
				const u32 hi = end < f.n ? f.seq_off[end] : tp.n_seq_units;
				if (hi > lo && hi - lo <= tp.seq_capacity_units) { units = hi - lo; mbar_expect_tx(bar, units * 16); bulk_g2s(staged, f.seq + (size_t) lo * 16, units * 16, bar); }
			}
			lo = __shfl_sync(0xFFFFFFFFu, lo, 0); units = __shfl_sync(0xFFFFFFFFu, units, 0);
		}
		fragment_inputs in;
		if (mine) in = fragment_inputs_of(f, i); // the columns of the fragment travel while the bulk copy is in flight
		if (units) { mbar_wait(bar, parity); parity ^= 1; }
		if (mine) {
			if (units) { in.seq0 = staged + (size_t) (f.seq_off[f.idx(i, 0)] - lo) * 16; in.seq1 = staged + (size_t) (f.seq_off[f.idx(i, 1)] - lo) * 16; }
			const u8 label = classify_sequences_group(g, p, f, an, i, in, counters, counters + 64);
			if (g.lane == 0) f.filter[i] = label;
		}
		__syncwarp(); // the warp's staging buffer is free again
	}
}
#endif

// test hook: (mismatches, compared bases) of the two alignments the mismatch rule walks, on the packed reference and base by base
struct mismatch_probe_fn {
	frag_view f; annot_view packed, plain; u32* out; // 8 per fragment
	ARB_HD void operator()(u32 i) const {
		const u32 n = f.n_aln[i], a0 = f.idx(i, 0), a1 = f.idx(i, 1), a2 = f.idx(i, 2);
		const u32 y = n == 2 ? a1 : a2; const bool rc = n == 3 && f.fwd(a2) != f.fwd(a1);
		u32* o = out + (size_t) i * 8;
		count_mismatches(f, packed, a0, f.sq(a0), f.seq_len[a0], false, o[0], o[1]);
		count_mismatches(f, packed, y, f.sq(a1), f.seq_len[a1], rc, o[2], o[3]);
		count_mismatches(f, plain, a0, f.sq(a0), f.seq_len[a0], false, o[4], o[5]);
		count_mismatches(f, plain, y, f.sq(a1), f.seq_len[a1], rc, o[6], o[7]);
	}
};
void engine::probe_mismatch_counts(u32* out) {
	if (!annot.assembly4_ok) throw arb_error("the packed reference is disabled (characters outside the nt16 alphabet)");
	dbuf<u32> d((size_t) frags.n * 8);
	annot_view plain = annot.view(); plain.assembly4 = 0;
	mismatch_probe_fn fn = {frags.view(), annot.view(), plain, d.ptr()};
	for_each(ex, frags.n, fn);
	d.download(ex, out, (size_t) frags.n * 8);
}

struct count_labels_fn {
	const u8* filter; u32* counts;
	ARB_HD void operator()(u32 i) const { atomic_add_u32(&counts[filter[i] < F_COUNT ? filter[i] : 0], 1); }
};

void engine::run_read_filters() {
	if (!has_contigs || !has_annotation) throw arb_error("arb_run_read_filters: contigs and annotation must be set first");
	const u32 n = frags.n;
	const read_filter_params p = make_filter_params();
	frag_view f = frags.view();
	stage_timer t_all(ex);
	{
	stage_timer t_dup(ex);
	if (p.enabled(F_duplicates)) {
		if (p.external_duplicate_marking) {
			dup_external_fn fn = {f};
			for_each(ex, n, fn);
		} else {
			dbuf<u64> k0(n); dbuf<u32> k1(n), slot(n), first(n); dbuf<u8> part(n);
			dup_key_fn kf = {f, k0.ptr(), k1.ptr(), part.ptr()};
			for_each(ex, n, kf);
			dup_key_ops ops = {k0.ptr(), k1.ptr()};
			group_min_index(ex, table, n, ops, part.ptr(), slot.ptr(), first.ptr());
			dup_mark_fn mf = {first.ptr(), part.ptr(), f.filter};
			for_each(ex, n, mf);
			ex.sync();
		}
	}
	timings.duplicates_ms = t_dup.stop();
	}
	{
		dbuf<u32> n_queued(1); dbuf<u8> needs(n);
		n_queued.zero(ex, 1);
		stage_timer t_cls(ex);
		stage_timer t_head(ex);
		cascade_head_fn hf = {p, f, annot.view(), frags.early.ptr(), needs.ptr(), n_queued.ptr()};
		for_each(ex, n, hf);
		timings.cascade_head_ms = t_head.stop();
		stage_timer t_seq(ex);
#ifdef ARB_DEVICE_BUILD
		if (n) {
			// shared memory per block: staging room for the tile's sequences + per group 64 counters and one word of dense codes per 8 bases (reads beyond 500 bases
			// are counted exactly by one lane and need no dense codes)
			const u32 len_cap = std::min<u32>(frags.max_seq_len, 1000);
			cascade_tile_params tp;
			tp.group_words = (64 + 2 * ((len_cap + 7) / 8) + 4) | 1; // odd: the groups' counters start in different banks
			const u32 units_per_read = ((frags.max_seq_len + 1) / 2 + 15) / 16;
			tp.seq_capacity_units = frags.canonical_seq_layout && (size_t) units_per_read * 2 * CASCADE_GROUPS * 16 <= 96 * 1024 ? units_per_read * 2 * CASCADE_GROUPS_PER_WARP : 0;
			tp.n_seq_units = (u32) (frags.n_seq_bytes / 16);
			const size_t shared_bytes = (size_t) tp.seq_capacity_units * 16 * (CASCADE_THREADS / 32) + (size_t) tp.group_words * 4 * CASCADE_GROUPS;
			if (shared_bytes != cascade_smem_bytes) { // function attributes and occupancy are per device: cached in the context
				ARB_CUDA_CHECK(cudaFuncSetAttribute(k_cascade_sequences, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) std::max<size_t>(shared_bytes, 48 * 1024)));
				int per_sm = 0, n_sm = 0;
				ARB_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_cascade_sequences, (int) CASCADE_THREADS, shared_bytes));
				ARB_CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
				cascade_resident_blocks = (u32) std::max(1, per_sm) * (u32) n_sm; cascade_smem_bytes = shared_bytes;
			}
			const u32 n_tiles = (n + CASCADE_GROUPS - 1) / CASCADE_GROUPS; // block-sized chunks of the warps' tiles
			const u32 grid = std::min<u32>(n_tiles, cascade_resident_blocks); // persistent: SM count x resident blocks per SM
			k_cascade_sequences<<<grid, CASCADE_THREADS, shared_bytes, ex.stream>>>(p, f, annot.view(), needs.ptr(), tp);
			ARB_CUDA_CHECK(cudaGetLastError());
			++stats().kernels;
		}
#else
		cascade_sequences_fn sf = {p, f, annot.view(), needs.ptr()};
		for_each_scratch<384>(ex, n, sf); // 64 counters + dense codes + predecessor masks of reads up to 1,000 bases
#endif
		timings.cascade_sequences_ms = t_seq.stop();
		timings.classify_ms = t_cls.stop();
		u32 q = 0; n_queued.download(ex, &q, 1);
		timings.cascade_queued = q;
		timings.cascade_algorithmic_bytes[0] = head_bytes;
		timings.cascade_algorithmic_bytes[1] = n ? (u64) ((double) sequence_bytes * q / n) : 0;
		timings.classify_algorithmic_bytes = timings.cascade_algorithmic_bytes[0] + timings.cascade_algorithmic_bytes[1];
	}
	timings.read_filters_ms = t_all.stop();
	ex.sync();
	filters_done = true;
}

void engine::get_fragment_filters(u8* filter_out, u8* early_out) {
	if (filter_out) frags.filter.download(ex, filter_out, frags.n);
	if (early_out) frags.early.download(ex, early_out, frags.n);
}

void engine::set_fragment_filters(const u8* filter) { frags.filter.upload(ex, filter, frags.n); ex.sync(); }

void engine::get_filter_counts(u32* counts) {
	label_counts.ensure(F_COUNT);
	label_counts.zero(ex, F_COUNT);
	count_labels_fn fn = {frags.filter.ptr(), label_counts.ptr()};
	for_each(ex, frags.n, fn);
	label_counts.download(ex, counts, F_COUNT);
}

} // namespace arb
