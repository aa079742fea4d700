// capi.cu -- the C ABI declared in include/arriba_b200.h: thin exception-to-status shims over arb::engine.
#include "engine.h"
#include <new>

using namespace arb;

struct arb_ctx { engine e; };
static std::string g_create_error;

// ---- page-locked host memory for the caller's columns -----------------------------------------------------------------------------------------------
// The host side builds its large columns in recycled blocks (host/ingest.h, host_block_get); in the CUDA library fresh blocks are page-locked, so that
// arb_push_chunk_begin/end copy them asynchronously at full PCIe speed. ARB_PINNED_HOST=0 keeps them pageable.
namespace arb { namespace host { void set_host_block_backend(void* (*alloc)(size_t), void (*release)(void*)); } }
static int g_host_memory_device = -1;
#ifdef ARB_DEVICE_BUILD
static void* pinned_alloc(size_t bytes) {
	if (g_host_memory_device >= 0) { int cur = -1; if (cudaGetDevice(&cur) != cudaSuccess || cur != g_host_memory_device) { if (cudaSetDevice(g_host_memory_device) != cudaSuccess) { cudaGetLastError(); return NULL; } } }
	void* p = NULL;
	if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return NULL; }
	return p;
}
static void pinned_free(void* p) { cudaFreeHost(p); }
namespace { struct install_pinned_backend { install_pinned_backend() { const char* s = getenv("ARB_PINNED_HOST"); if (!s || atoi(s) != 0) arb::host::set_host_block_backend(pinned_alloc, pinned_free); } } g_install_pinned_backend; }
#endif

#ifdef ARB_DEVICE_BUILD
#define ARB_BIND_DEVICE(ctx) ARB_CUDA_CHECK(cudaSetDevice((ctx)->e.device));
#else
#define ARB_BIND_DEVICE(ctx)
#endif
#define ARB_API_BEGIN(ctx) if (!(ctx)) return 2; try { ARB_BIND_DEVICE(ctx)
#define ARB_API_END(ctx) } catch (const std::exception& x) { (ctx)->e.last_error = x.what(); return 1; } catch (...) { (ctx)->e.last_error = "unknown error"; return 1; } return 0;

extern "C" {

const char* arb_backend(void) {
#ifdef ARB_DEVICE_BUILD
	return "cuda-sm_100a";
#else
	return "hostsim-TEST-ONLY";
#endif
}

uint64_t arb_kernel_launches(void) { return stats().kernels; }

int arb_ctx_create(arb_ctx** out, int device) {
	if (!out) return 2;
	*out = NULL;
	try {
#ifdef ARB_DEVICE_BUILD
		int count = 0;
		cudaError_t e = cudaGetDeviceCount(&count);
		if (e != cudaSuccess || count == 0) throw arb_error(std::string("no usable CUDA device (") + cudaGetErrorString(e) + "); arriba-b200 has no CPU fallback");
		if (device < 0 || device >= count) throw arb_error("device index out of range");
		ARB_CUDA_CHECK(cudaSetDevice(device));
		cudaDeviceProp prop;
		ARB_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
		if (prop.major < 10) throw arb_error(std::string("device '") + prop.name + "' is not sm_100-class; this build targets sm_100a only");
#else
		(void) device;
#endif
#ifdef ARB_DEVICE_BUILD
		cudaSetDeviceFlags(cudaDeviceLmemResizeToMax); cudaGetLastError(); // keep the local-memory arena of the recursive re-alignment kernels between launches (best effort)
		ARB_CUDA_CHECK(cudaDeviceSetLimit(cudaLimitStackSize, 16 * 1024)); // realign() recurses at splice sites and at one deletion (mismap_hd.h)
#endif
		*out = new arb_ctx();
		(*out)->e.device = device;
	} catch (const std::exception& x) { g_create_error = x.what(); return 1; }
	return 0;
}

void arb_ctx_destroy(arb_ctx* ctx) {
	if (!ctx) return;
#ifdef ARB_DEVICE_BUILD
	cudaSetDevice(ctx->e.device);
#endif
	delete ctx; // device blocks go back to the pool, not to the driver: the next context on this device reuses them
}
void arb_release_device_memory(void) { pool_trim(); }
void arb_set_host_memory_device(int device) { g_host_memory_device = device; }
const char* arb_last_error(arb_ctx* ctx) { return ctx ? ctx->e.last_error.c_str() : g_create_error.c_str(); }

void arb_default_params(arb_params* p) { if (p) default_params(*p); }
int arb_set_params(arb_ctx* ctx, const arb_params* p) { ARB_API_BEGIN(ctx) ctx->e.set_params(*p); ARB_API_END(ctx) }
int arb_set_contigs(arb_ctx* ctx, const arb_contigs* c) { ARB_API_BEGIN(ctx) ctx->e.set_contigs(*c); ARB_API_END(ctx) }
int arb_set_annotation(arb_ctx* ctx, const arb_annotation* a) { ARB_API_BEGIN(ctx) ctx->e.set_annotation(*a); ARB_API_END(ctx) }
int arb_set_contig_flags(arb_ctx* ctx, const uint8_t* flags, uint32_t n) { ARB_API_BEGIN(ctx) ctx->e.set_contig_flags(flags, n); ARB_API_END(ctx) }
int arb_push_chunk(arb_ctx* ctx, const arb_soa_chunk* c) { ARB_API_BEGIN(ctx) ctx->e.push_chunk(*c); ARB_API_END(ctx) }
int arb_push_chunk_begin(arb_ctx* ctx, const arb_soa_chunk* c) { ARB_API_BEGIN(ctx) ctx->e.push_chunk_begin(*c); ARB_API_END(ctx) }
int arb_push_chunk_end(arb_ctx* ctx, const arb_soa_chunk* c) { ARB_API_BEGIN(ctx) ctx->e.push_chunk_end(*c); ARB_API_END(ctx) }
int arb_bam_scan(arb_ctx* ctx, const uint8_t* chunk, uint64_t bytes, uint64_t first, int32_t n_ref, uint32_t n_lists, uint64_t* consumed, uint32_t* n_records, uint32_t* list_begin, uint32_t* record_offsets, uint32_t* malformed) {
	ARB_API_BEGIN(ctx) u64 c = 0; ctx->e.bam_scan(chunk, bytes, first, n_ref, n_lists, &c, n_records, list_begin, record_offsets, malformed); *consumed = c; ARB_API_END(ctx)
}
int arb_build_fragment_table(arb_ctx* ctx, const arb_ingest_pool* pools, uint32_t n_pools, arb_fragment_table_sizes* sizes) {
	ARB_API_BEGIN(ctx) if (!sizes) throw arb_error("arb_build_fragment_table: sizes is NULL"); memset(sizes, 0, sizeof(*sizes)); ctx->e.build_fragment_table(pools, n_pools, *sizes); ARB_API_END(ctx)
}
uint32_t arb_fragment_table_tie_rounds(arb_ctx* ctx) { return ctx ? ctx->e.tie_rounds : 0; }
int arb_get_fragment_table(arb_ctx* ctx, const arb_fragment_columns* out) { ARB_API_BEGIN(ctx) if (!out) throw arb_error("arb_get_fragment_table: out is NULL"); ctx->e.get_fragment_table(*out); ARB_API_END(ctx) }
int arb_annotate_pass1(arb_ctx* ctx, const uint8_t* aflags, int32_t strandedness, uint32_t* n_dummy) { ARB_API_BEGIN(ctx) const uint32_t k = ctx->e.annotate_pass1(aflags, strandedness); if (n_dummy) *n_dummy = k; ARB_API_END(ctx) }
int arb_get_dummy_genes(arb_ctx* ctx, uint16_t* contig, int32_t* start, int32_t* end) { ARB_API_BEGIN(ctx) ctx->e.get_dummy_genes(contig, start, end); ARB_API_END(ctx) }
int arb_annotate_pass2(arb_ctx* ctx, uint64_t* n_gene_ids) { ARB_API_BEGIN(ctx) const uint64_t k = ctx->e.annotate_pass2(); if (n_gene_ids) *n_gene_ids = k; ARB_API_END(ctx) }
int arb_get_annotation_columns(arb_ctx* ctx, uint8_t* aflags, uint32_t* genes_off, uint16_t* genes_cnt, uint32_t* genes) { ARB_API_BEGIN(ctx) ctx->e.get_annotation_columns(aflags, genes_off, genes_cnt, genes); ARB_API_END(ctx) }
int arb_run_read_filters(arb_ctx* ctx) { ARB_API_BEGIN(ctx) ctx->e.run_read_filters(); ARB_API_END(ctx) }
int arb_get_fragment_filters(arb_ctx* ctx, uint8_t* f, uint8_t* early) { ARB_API_BEGIN(ctx) ctx->e.get_fragment_filters(f, early); ARB_API_END(ctx) }
int arb_set_fragment_filters(arb_ctx* ctx, const uint8_t* f) { ARB_API_BEGIN(ctx) ctx->e.set_fragment_filters(f); ARB_API_END(ctx) }
int arb_get_filter_counts(arb_ctx* ctx, uint32_t counts[ARB_N_FILTERS]) { ARB_API_BEGIN(ctx) ctx->e.get_filter_counts(counts); ARB_API_END(ctx) }
int arb_find_fusions(arb_ctx* ctx, int32_t max_mate_gap) { ARB_API_BEGIN(ctx) ctx->e.find_fusions(max_mate_gap); ARB_API_END(ctx) }
int arb_candidates_size(arb_ctx* ctx, uint32_t* n, uint64_t* n1, uint64_t* n2, uint64_t* nd) {
	ARB_API_BEGIN(ctx)
	if (n) *n = ctx->e.cands.n; if (n1) *n1 = ctx->e.cands.n_list1; if (n2) *n2 = ctx->e.cands.n_list2; if (nd) *nd = ctx->e.cands.n_listd;
	ARB_API_END(ctx)
}
int arb_get_candidates(arb_ctx* ctx, arb_candidates* out) { ARB_API_BEGIN(ctx) ctx->e.get_candidates(*out); ARB_API_END(ctx) }
int arb_set_candidate_state(arb_ctx* ctx, const uint8_t* f, const uint32_t* s1, const uint32_t* s2, const uint32_t* dm, const float* ev) { ARB_API_BEGIN(ctx) ctx->e.set_candidate_state(f, s1, s2, dm, ev); ARB_API_END(ctx) }
int arb_get_candidate_filters(arb_ctx* ctx, uint8_t* f) { ARB_API_BEGIN(ctx) ctx->e.cands.filter.download(ctx->e.ex, f, ctx->e.cands.n); ARB_API_END(ctx) }
int arb_get_candidate_state(arb_ctx* ctx, uint8_t* f, uint32_t* s1, uint32_t* s2, uint32_t* dm, float* ev) { ARB_API_BEGIN(ctx) ctx->e.get_candidate_state(f, s1, s2, dm, ev); ARB_API_END(ctx) }
int arb_set_candidate_lists(arb_ctx* ctx, const uint32_t* l1o, const uint32_t* l1, const uint32_t* l2o, const uint32_t* l2) { ARB_API_BEGIN(ctx) ctx->e.set_candidate_lists(l1o, l1, l2o, l2); ARB_API_END(ctx) }
int arb_merge_adjacent(arb_ctx* ctx, int32_t max_distance, uint32_t* n) { ARB_API_BEGIN(ctx) uint32_t k = ctx->e.merge_adjacent(max_distance); if (n) *n = k; ARB_API_END(ctx) }
int arb_get_merge_log(arb_ctx* ctx, uint32_t* triples, uint32_t n) { ARB_API_BEGIN(ctx) ctx->e.get_merge_log(triples, n); ARB_API_END(ctx) }
int arb_estimate_evalues(arb_ctx* ctx, const arb_evalue_inputs* in) { ARB_API_BEGIN(ctx) ctx->e.estimate_evalues(*in); ARB_API_END(ctx) }
int arb_select_best(arb_ctx* ctx, uint32_t* remaining) { ARB_API_BEGIN(ctx) const uint32_t r = ctx->e.select_best(); if (remaining) *remaining = r; ARB_API_END(ctx) }
int arb_evalue_tallies(arb_ctx* ctx, uint32_t out[11]) { ARB_API_BEGIN(ctx) ctx->e.evalue_tallies(out); ARB_API_END(ctx) }
int arb_filter_simple(arb_ctx* ctx, int32_t stage, float exonic_fraction, int32_t min_support, uint32_t* remaining) { ARB_API_BEGIN(ctx) const uint32_t r = ctx->e.filter_simple(stage, exonic_fraction, min_support); if (remaining) *remaining = r; ARB_API_END(ctx) }
int arb_filter_relative_support(arb_ctx* ctx, float cutoff) { ARB_API_BEGIN(ctx) ctx->e.filter_relative_support(cutoff); ARB_API_END(ctx) }
int arb_set_coverage(arb_ctx* ctx, const uint16_t* const* cov, const uint64_t* n_windows, uint32_t n_contigs) { ARB_API_BEGIN(ctx) std::vector<u64> w(n_windows, n_windows + n_contigs); ctx->e.set_coverage(cov, w.data(), n_contigs); ARB_API_END(ctx) }
int arb_reads_by_gene(arb_ctx* ctx, uint32_t* out) { ARB_API_BEGIN(ctx) ctx->e.reads_by_gene(out); ARB_API_END(ctx) }
int arb_filter_in_vitro(arb_ctx* ctx, const uint32_t* reads, uint32_t n_genes, uint32_t threshold, const uint64_t* pairs, uint64_t n_pairs) { ARB_API_BEGIN(ctx) ctx->e.filter_in_vitro(reads, n_genes, threshold, (const u64*) pairs, n_pairs); ARB_API_END(ctx) }
int arb_spliced_support(arb_ctx* ctx, const uint32_t* reads, uint32_t n_genes, uint32_t threshold, uint32_t* out) { ARB_API_BEGIN(ctx) ctx->e.spliced_support(reads, n_genes, threshold, out); ARB_API_END(ctx) }
int arb_replay_insertion_order(arb_ctx* ctx, const uint32_t* phase_start, const uint64_t* phase_buckets, uint32_t n_phases, uint32_t* order_out, uint32_t* rank_out) { ARB_API_BEGIN(ctx) ctx->e.replay_insertion_order(phase_start, (const u64*) phase_buckets, n_phases, order_out, rank_out); ARB_API_END(ctx) }
int arb_partner_counts(arb_ctx* ctx, int32_t* out) { ARB_API_BEGIN(ctx) ctx->e.partner_counts(out); ARB_API_END(ctx) }
int arb_set_row_texts(arb_ctx* ctx, const arb_row_texts* t) { ARB_API_BEGIN(ctx) if (!t) throw arb_error("null tables"); ctx->e.set_row_texts(*t); ARB_API_END(ctx) }
int arb_format_discarded_rows(arb_ctx* ctx, const uint8_t* confidence, uint64_t* n_rows, uint64_t* n_bytes) { ARB_API_BEGIN(ctx) u64 r = 0, b = 0; ctx->e.format_discarded_rows(confidence, &r, &b); *n_rows = r; *n_bytes = b; ARB_API_END(ctx) }
int arb_get_row_text(arb_ctx* ctx, char* out) { ARB_API_BEGIN(ctx) ctx->e.get_row_text(out); ARB_API_END(ctx) }
int arb_build_consensus(arb_ctx* ctx, const uint32_t* candidates, uint32_t n_rows, arb_consensus_info* info) { ARB_API_BEGIN(ctx) ctx->e.build_consensus(candidates, n_rows, *info); ARB_API_END(ctx) }
int arb_get_consensus(arb_ctx* ctx, uint32_t* seq_off, uint32_t* pos_off, uint32_t* clip_off, uint8_t* verdict, uint32_t* non_template, char* seq, int32_t* pos, char* clip) {
	ARB_API_BEGIN(ctx) ctx->e.get_consensus(seq_off, pos_off, clip_off, verdict, non_template, seq, pos, clip); ARB_API_END(ctx)
}
int arb_filter_multimappers(arb_ctx* ctx) { ARB_API_BEGIN(ctx) ctx->e.filter_multimappers(); ARB_API_END(ctx) }
int arb_set_splice_sites(arb_ctx* ctx, const uint32_t* off, const int32_t* sites) { ARB_API_BEGIN(ctx) ctx->e.set_splice_sites(off, sites); ARB_API_END(ctx) }
int arb_build_kmer_index(arb_ctx* ctx, const uint32_t* contig, const int32_t* start, const int32_t* end, uint32_t n, uint32_t nc, uint64_t* n_indexed) { ARB_API_BEGIN(ctx) uint64_t k = ctx->e.build_kmer_index(contig, start, end, n, nc); if (n_indexed) *n_indexed = k; ARB_API_END(ctx) }
int arb_kmer_index_digest(arb_ctx* ctx, uint64_t* kmers, uint64_t* positions, uint64_t* checksum, uint32_t nc) { ARB_API_BEGIN(ctx) ctx->e.kmer_index_digest(kmers, positions, checksum, nc); ARB_API_END(ctx) }
int arb_homolog_pairs(arb_ctx* ctx, const uint32_t* ga, const uint32_t* gb, uint32_t n, uint8_t* out) { ARB_API_BEGIN(ctx) ctx->e.homolog_pairs(ga, gb, n, out); ARB_API_END(ctx) }
int arb_filter_mismappers(arb_ctx* ctx, int32_t max_mate_gap, uint64_t* n) { ARB_API_BEGIN(ctx) uint64_t k = ctx->e.filter_mismappers(max_mate_gap); if (n) *n = k; ARB_API_END(ctx) }
int arb_exchange_header(arb_ctx* ctx, int group, uint64_t* header, uint32_t* n_words) {
	ARB_API_BEGIN(ctx) std::vector<u64> h; ctx->e.exchange_header(group, h); if (h.size() > 16) throw arb_error("exchange header too long"); for (size_t k = 0; k < h.size(); ++k) header[k] = h[k]; *n_words = (uint32_t) h.size(); ARB_API_END(ctx)
}
int arb_exchange_prepare(arb_ctx* ctx, int group, const uint64_t* header, uint32_t n_words) { ARB_API_BEGIN(ctx) ctx->e.exchange_prepare(group, header, n_words); ARB_API_END(ctx) }
int arb_exchange_buffers(arb_ctx* ctx, int group, void** ptrs, uint64_t* bytes, uint32_t* n) {
	ARB_API_BEGIN(ctx) std::vector<exchange_buffer> b; ctx->e.exchange_buffers(group, b); if (b.size() > *n) throw arb_error("arb_exchange_buffers: capacity too small"); for (size_t k = 0; k < b.size(); ++k) { ptrs[k] = b[k].p; bytes[k] = b[k].bytes; } *n = (uint32_t) b.size(); ARB_API_END(ctx)
}
int arb_exchange_commit(arb_ctx* ctx, int group) { ARB_API_BEGIN(ctx) ctx->e.exchange_commit(group); ARB_API_END(ctx) }
int arb_set_work_partition(arb_ctx* ctx, const uint32_t* keys, const uint8_t* owner, uint32_t n_keys, int part, int parts) { ARB_API_BEGIN(ctx) ctx->e.set_work_partition(keys, owner, n_keys, part, parts); ARB_API_END(ctx) }
int arb_candidates_export(arb_ctx* ctx, void** blob, uint64_t* bytes, uint64_t sizes[4]) { ARB_API_BEGIN(ctx) u64 s[4]; u64 b = 0; ctx->e.candidates_export(blob, &b, s); *bytes = b; for (int k = 0; k < 4; ++k) sizes[k] = s[k]; ARB_API_END(ctx) }
int arb_candidates_import(arb_ctx* ctx, const void* all_blobs, uint64_t stride, const uint64_t* sizes, uint32_t n_parts) { ARB_API_BEGIN(ctx) std::vector<u64> s(sizes, sizes + 4 * (size_t) n_parts); ctx->e.candidates_import(all_blobs, stride, s.data(), n_parts); ARB_API_END(ctx) }
int arb_swaps_buffer(arb_ctx* ctx, void** p, uint64_t* bytes) { ARB_API_BEGIN(ctx) u64 b = 0; ctx->e.swaps_buffer(p, &b); *bytes = b; ARB_API_END(ctx) }
int arb_swaps_apply(arb_ctx* ctx) { ARB_API_BEGIN(ctx) ctx->e.swaps_apply(); ARB_API_END(ctx) }
int arb_filter_mismappers_part(arb_ctx* ctx, int32_t max_mate_gap, int part, int parts, void** verdicts, uint64_t* bytes) { ARB_API_BEGIN(ctx) u64 b = 0; ctx->e.filter_mismappers_part(max_mate_gap, part, parts, verdicts, &b); *bytes = b; ARB_API_END(ctx) }
int arb_filter_mismappers_finish(arb_ctx* ctx, uint64_t* n) { ARB_API_BEGIN(ctx) const uint64_t k = ctx->e.filter_mismappers_finish(); if (n) *n = k; ARB_API_END(ctx) }
int arb_get_timings(arb_ctx* ctx, arb_timings* out) { ARB_API_BEGIN(ctx) *out = ctx->e.timings; ARB_API_END(ctx) }
int arb_selftest_mismatch_counts(arb_ctx* ctx, uint32_t* out) { ARB_API_BEGIN(ctx) ctx->e.probe_mismatch_counts(out); ARB_API_END(ctx) } // tests only, not declared in the public header
int arb_set_candidates(arb_ctx* ctx, const arb_candidates* c) { ARB_API_BEGIN(ctx) if (!c) throw arb_error("null table"); ctx->e.set_candidates(*c); ARB_API_END(ctx) }
int arb_apply_slot_swaps(arb_ctx* ctx, const uint8_t* swapped) { ARB_API_BEGIN(ctx) ctx->e.apply_slot_swaps(swapped); ARB_API_END(ctx) }
int arb_get_candidate_first_fragments(arb_ctx* ctx, uint32_t* out) { ARB_API_BEGIN(ctx) ctx->e.get_first_fragments(out); ARB_API_END(ctx) }
int arb_get_slot_swaps(arb_ctx* ctx, uint8_t* out) { ARB_API_BEGIN(ctx) ctx->e.get_slot_swaps(out); ARB_API_END(ctx) }

} // extern "C"
