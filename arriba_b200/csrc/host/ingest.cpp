// ingest.cpp -- see ingest.h. BGZF blocks are inflated in parallel, records are sharded by read name over worker threads
// (every alignment of a read name is handled by the same worker, so mate collation and "first insertion wins" stay local),
// and the fragments are finally ordered by name on the device (csrc/fragtable.cu), which is the order every later stage relies on.
#include "ingest.h"
#include "../../../include/arriba_b200.h"
#include <set>
#include "../annot_hd.h"
#include <zlib.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <algorithm>
#include <chrono>
#include <cstring>
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <stdexcept>
#include <thread>
#include <mutex>
#include <unordered_map>

namespace arb { namespace host {

// ------------------------------------------------------------------------------------------- recycled host blocks (ingest.h)
namespace {
struct host_block_pool {
	std::mutex lock; std::vector<std::pair<size_t, void*> > free_blocks; size_t held;
	std::set<void*> from_backend; // blocks obtained from the backend (page-locked memory in the CUDA library): they go back through it
	host_block_pool(): held(0) {}
};
void* (*g_backend_alloc)(size_t) = NULL; void (*g_backend_free)(void*) = NULL;
host_block_pool& block_pool() { static host_block_pool* p = new host_block_pool(); return *p; } // never destroyed: blocks may be returned during static destruction
}
void* host_block_get(size_t bytes, size_t& granted) {
	granted = bytes;
	host_block_pool& pool = block_pool();
	{
		std::lock_guard<std::mutex> g(pool.lock);
		for (size_t k = pool.free_blocks.size(); k-- > 0; ) if (pool.free_blocks[k].first == bytes) {
			void* p = pool.free_blocks[k].second; pool.free_blocks[k] = pool.free_blocks.back(); pool.free_blocks.pop_back(); pool.held -= bytes; return p;
		}
	}
	if (g_backend_alloc) { // page-locked: the columns built in such blocks are copied to the device asynchronously at full PCIe speed, and the blocks are recycled
		void* p = g_backend_alloc(bytes);
		if (p) { std::lock_guard<std::mutex> g(pool.lock); pool.from_backend.insert(p); return p; }
	}
	return malloc(bytes);
}
static void release_block(host_block_pool& pool, void* p) { // pool.lock held
	std::set<void*>::iterator it = pool.from_backend.find(p);
	if (it != pool.from_backend.end()) { pool.from_backend.erase(it); g_backend_free(p); } else free(p);
}
void host_block_put(void* p, size_t granted) {
	host_block_pool& pool = block_pool();
	std::lock_guard<std::mutex> g(pool.lock);
	if (pool.held + granted <= ((size_t) 64 << 30)) { pool.free_blocks.push_back(std::make_pair(granted, p)); pool.held += granted; return; }
	release_block(pool, p);
}
void host_block_trim() {
	host_block_pool& pool = block_pool();
	std::lock_guard<std::mutex> g(pool.lock);
	for (size_t k = 0; k < pool.free_blocks.size(); ++k) release_block(pool, pool.free_blocks[k].second);
	pool.free_blocks.clear(); pool.held = 0;
}
void set_host_block_backend(void* (*alloc)(size_t), void (*release)(void*)) { g_backend_alloc = alloc; g_backend_free = release; }

static void fail(const std::string& m) { throw std::runtime_error(m); }
// Tables of hundreds of megabytes that are visited all over (name slots, fragments, alignments, coverage windows): on 4 KiB pages nearly every visit also misses
// the TLB. Where the kernel offers transparent huge pages on request (THP "madvise"), ask for them; elsewhere the call does nothing.
static void advise_huge(const void* p, size_t bytes) {
#ifdef MADV_HUGEPAGE
	const size_t huge = (size_t) 2 << 20;
	static const bool enabled = getenv("ARB_HUGE_PAGES") == NULL || atoi(getenv("ARB_HUGE_PAGES")) != 0;
	if (!enabled || p == NULL || bytes < 4 * huge) return;
	const uintptr_t lo = ((uintptr_t) p + huge - 1) & ~(uintptr_t) (huge - 1), hi = ((uintptr_t) p + bytes) & ~(uintptr_t) (huge - 1);
	if (hi > lo) madvise((void*) lo, hi - lo, MADV_HUGEPAGE);
#else
	(void) p; (void) bytes;
#endif
}
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

enum { BF_PAIRED = 1, BF_PROPER = 2, BF_UNMAP = 4, BF_MUNMAP = 8, BF_REVERSE = 16, BF_READ1 = 64, BF_SECONDARY = 256, BF_DUP = 1024, BF_SUPPLEMENTARY = 2048 };

static inline u32 rd32(const u8* p) { u32 v; memcpy(&v, p, 4); return v; }
static inline u16 rd16(const u8* p) { u16 v; memcpy(&v, p, 2); return v; }

// ------------------------------------------------------------------------------------------- coverage
void coverage_windows::resize(const refdata& ref) {
	const size_t nc = ref.contig_ids.size();
	coverage.resize(nc); starts.resize(nc); ends.resize(nc);
	for (size_t c = 0; c < nc; ++c) if (ref.has_sequence((u32) c)) {
		const size_t w = ref.seq_len[c] / 20 + 2;
		if (coverage[c].size() < w) { coverage[c].reserve(w); advise_huge(coverage[c].data(), w * sizeof(coverage[c][0])); coverage[c].resize(w, 0); starts[c].resize(w, 0); ends[c].resize(w, 0); }
	}
}
bool coverage_windows::fragment_starts_here(u32 contig, i32 start, i32 end) const {
	if (contig >= starts.size()) return false;
	for (int w = start / 20 + 1; w <= end / 20; ++w) { if ((u32) w >= starts[contig].size()) return false; if (starts[contig][w]) return true; }
	return false;
}
bool coverage_windows::fragment_ends_here(u32 contig, i32 start, i32 end) const {
	if (contig >= ends.size()) return false;
	for (int w = start / 20; w < end / 20; ++w) { if ((u32) w >= ends[contig].size()) return false; if (ends[contig][w]) return true; }
	return false;
}
int coverage_windows::get_coverage(u32 contig, i32 position, u32 direction) const {
	if (contig >= coverage.size() || coverage[contig].empty()) return -1;
	if (direction == UPSTREAM) return position < 20 ? 0 : coverage[contig][position / 20 - 1];
	return coverage[contig][position / 20 + 1];
}

// ------------------------------------------------------------------------------------------- parsed BAM record
struct rec_t {
	const u8* base; u32 size;       // record body (after block_size)
	i32 tid, pos; u16 flag; u32 n_cigar; i32 l_seq; u32 l_qname;
	const char* qname; const u8* cigar_raw; const u8* seq; const u8* aux; const u8* aux_end;
	bool valid() const { return base != NULL; }
	bool reverse() const { return flag & BF_REVERSE; }
	u32 cig(u32 k) const { return rd32(cigar_raw + 4 * k); }
	i32 ref_len(u32 n_ops) const { i64 l = 0; for (u32 k = 0; k < n_ops; ++k) { u32 c = cig(k), o = c & 15; if (o == C_M || o == C_D || o == C_N || o == C_EQ || o == C_X) l += c >> 4; } return (i32) l; }
	i32 query_len(u32 n_ops) const { i64 l = 0; for (u32 k = 0; k < n_ops; ++k) { u32 c = cig(k), o = c & 15; if (o == C_M || o == C_I || o == C_S || o == C_EQ || o == C_X) l += c >> 4; } return (i32) l; }
	i32 endpos() const { i32 r = (flag & BF_UNMAP) ? 0 : ref_len(n_cigar); if (r == 0) r = 1; return pos + r; }
	u32 base_code(u32 i) const { return nt16_at(seq, i); }
};

static bool parse_record(const u8* p, u32 size, rec_t& r) {
	if (size < 32) return false;
	r.base = p; r.size = size;
	r.tid = (i32) rd32(p); r.pos = (i32) rd32(p + 4); r.l_qname = p[8]; r.n_cigar = rd16(p + 12); r.flag = rd16(p + 14); r.l_seq = (i32) rd32(p + 16);
	const u64 need = 32ull + r.l_qname + 4ull * r.n_cigar + ((u64) r.l_seq + 1) / 2 + (u64) r.l_seq;
	if (need > size || r.l_qname == 0) return false;
	r.qname = (const char*) p + 32; r.cigar_raw = p + 32 + r.l_qname; r.seq = r.cigar_raw + 4 * r.n_cigar;
	r.aux = r.seq + (r.l_seq + 1) / 2 + r.l_seq; r.aux_end = p + size;
	return true;
}

static const u8* find_aux(const rec_t& r, char a, char b) { // returns pointer to the type byte
	const u8* s = r.aux;
	while (s + 3 <= r.aux_end) {
		const bool hit = s[0] == (u8) a && s[1] == (u8) b;
		const u8* v = s + 2; const u8 t = v[0]; const u8* next;
		switch (t) {
			case 'A': case 'c': case 'C': next = v + 2; break;
			case 's': case 'S': next = v + 3; break;
			case 'i': case 'I': case 'f': next = v + 5; break;
			case 'd': next = v + 9; break;
			case 'Z': case 'H': next = v + 1; while (next < r.aux_end && *next) ++next; ++next; break;
			case 'B': {
				if (v + 6 > r.aux_end) return NULL;
				const u8 st = v[1]; const u32 n = rd32(v + 2);
				const u32 sz = (st == 'c' || st == 'C') ? 1 : (st == 's' || st == 'S') ? 2 : 4;
				next = v + 6 + (u64) sz * n; break;
			}
			default: return NULL;
		}
		if (next > r.aux_end) return NULL; // truncated field: its payload lies past the record (htslib reports corrupted aux data and returns no tag)
		if (hit) return v;
		s = next;
	}
	return NULL;
}
static i64 aux_int(const u8* v) {
	switch (v[0]) {
		case 'c': return (int8_t) v[1]; case 'C': return v[1]; case 's': return (int16_t) rd16(v + 1); case 'S': return rd16(v + 1);
		case 'i': return (i32) rd32(v + 1); case 'I': return rd32(v + 1); default: return 0;
	}
}

// paired-end reads must be clipped at the outer end of the fragment (read_chimeric_alignments.cpp:511-522)
static bool clipped_at_correct_end(const rec_t& r) {
	if (!(r.flag & BF_PAIRED)) return true;
	const bool fwd = !r.reverse();
	const u32 k = (r.flag & BF_SUPPLEMENTARY) ? (fwd ? r.n_cigar - 1 : 0) : (fwd ? 0 : r.n_cigar - 1);
	const u32 op = r.cig(k) & 15;
	return op == C_S || op == C_H;
}

// ------------------------------------------------------------------------------------------- per-worker fragment store
// the records of the pools that arb_build_fragment_table turns into the fragment table on the device
typedef arb_pool_alignment aln_build;
typedef arb_pool_fragment frag_build;

struct name_hash { size_t operator()(const std::string& s) const { u64 h = 1469598103934665603ULL; for (size_t i = 0; i < s.size(); ++i) { h ^= (u8) s[i]; h *= 1099511628211ULL; } return (size_t) h; } };

struct worker {
	refdata* ref; const ingest_options* opt; const std::vector<u16>* tid_to_contig; const std::vector<u8>* interesting_contig; const std::vector<u8>* viral_contig;
	annot_view an;
	// append-only pools, page-locked (host blocks of the CUDA library): they are copied to the device as they are when the record loop ends
	column<char> names; column<u32> cigars; column<u8> seqs; column<aln_build> alns; column<frag_build> frags;
	std::vector<u32> name_slots; // open-addressing index of `frags` by name: fragment id + 1, 0 = empty; names are compared in the `names` pool
	std::unordered_map<std::string, std::vector<u8>, name_hash> pending; // first mate of a proper pair, waiting for the second
	coverage_windows* cov; // shared by all workers: saturating counters and flags are updated atomically, the result does not depend on the order
	u64 mapped_reads, malformed, missing_hi, records; std::vector<u64> viral_reads; bool no_chimeric;
	std::string key, clip_chars, waiting_key; const u8* waiting_ptr; u32 waiting_size; u32 last_fragment;
	void park_waiting() { if (waiting_ptr) { pending.emplace(waiting_key, std::vector<u8>(waiting_ptr, waiting_ptr + waiting_size)); waiting_ptr = NULL; } } // before the chunk buffer is recycled
	worker(): cov(NULL), waiting_ptr(NULL), waiting_size(0), last_fragment(0xFFFFFFFFu), mapped_reads(0), malformed(0), missing_hi(0), records(0), no_chimeric(true), key_hash_hint(0) {}
	// A worker's pools are gigabytes that a sample touches for the first time page by page (a tenth of the ingest's CPU time went into those faults, tools/hostprof
	// on the GPU box): the workers of a finished sample are kept for the next one -- contents dropped, memory kept (arb_release_host_memory gives it back).
	void recycle() {
		names.clear(); cigars.clear(); seqs.clear(); alns.clear(); frags.clear(); pending.clear(); viral_reads.clear();
		std::fill(name_slots.begin(), name_slots.end(), 0u);
		ref = NULL; opt = NULL; tid_to_contig = NULL; interesting_contig = NULL; viral_contig = NULL; cov = NULL;
		mapped_reads = malformed = missing_hi = records = 0; no_chimeric = true; waiting_ptr = NULL; waiting_size = 0; last_fragment = 0xFFFFFFFFu; key_hash_hint = 0;
		key.clear(); clip_chars.clear(); waiting_key.clear();
	}

	u32 fragment(const std::string& name, bool* created = NULL, u64 hashed = 0) {
		// the records of one fragment follow each other in a collated BAM: remember the last answer before walking the table
		if (last_fragment != 0xFFFFFFFFu) { const frag_build& f = frags[last_fragment]; if (f.name_len == name.size() && memcmp(names.data() + f.name_off, name.data(), name.size()) == 0) { if (created) *created = false; return last_fragment; } }
		const u32 id = fragment_lookup(name, created, hashed);
		last_fragment = id;
		return id;
	}
	// Look-ahead of the record loop (read_chimeric_alignments below): the table walk of a record's fragment -- name slot, fragment, its name and last alignment --
	// is a chain of cache misses in tables of gigabytes. The loop computes the key hash of the record five steps ahead and requests the links of the chain one
	// step apart, so that process() finds them in the cache. Requests only: nothing here changes what process() does.
	u64 key_hash_hint; // hash of the key of the record process() is about to see (0: none)
	static u64 key_hash(const char* name, size_t n_name, i64 hit_index) { // FNV-1a over "<qname>,<HI>", folded like fragment_lookup does
		u64 h = 1469598103934665603ULL;
		for (size_t i = 0; i < n_name; ++i) { h ^= (u8) name[i]; h *= 1099511628211ULL; }
		h ^= (u8) ','; h *= 1099511628211ULL;
		char digits[24]; int n = 0; u64 v = hit_index < 0 ? 0 - (u64) hit_index : (u64) hit_index; do { digits[n++] = (char) ('0' + v % 10); v /= 10; } while (v);
		if (hit_index < 0) { h ^= (u8) '-'; h *= 1099511628211ULL; }
		while (n > 0) { h ^= (u8) digits[--n]; h *= 1099511628211ULL; }
		h ^= h >> 29;
		return h; // 0 (one key in 2^64) reads as "no hint": fragment_lookup then hashes the key itself
	}
	u64 ahead_hash(const u8* p, u32 size) { // the key hash of a record that has not been processed yet; also asks for its coverage windows
		rec_t r;
		if (!parse_record(p, size, r)) return 0;
		if ((r.flag & BF_UNMAP) || ((r.flag & BF_PAIRED) && (r.flag & BF_MUNMAP))) return 0;
		i64 hit_index = 1;
		const u8* hi = find_aux(r, 'H', 'I');
		if (hi) hit_index = aux_int(hi); else if (r.flag & BF_SECONDARY) return 0;
		if (r.tid >= 0 && (size_t) r.tid < tid_to_contig->size() && !(r.flag & BF_SUPPLEMENTARY)) {
			const u32 contig = (*tid_to_contig)[r.tid];
			if (contig < cov->coverage.size() && !cov->coverage[contig].empty()) { const size_t w = (size_t) (r.pos < 0 ? 0 : r.pos) / 20; if (w < cov->coverage[contig].size()) { __builtin_prefetch(&cov->coverage[contig][w], 1); __builtin_prefetch(&cov->coverage[contig][std::min(w + 5, cov->coverage[contig].size() - 1)], 1); } }
		}
		const u64 h = key_hash(r.qname, strnlen(r.qname, r.l_qname), hit_index);
		if (!name_slots.empty()) __builtin_prefetch(&name_slots[(size_t) h & (name_slots.size() - 1)]);
		return h;
	}
	void ahead_fragment(u64 h) const { if (h && !name_slots.empty()) { const u32 id = name_slots[(size_t) h & (name_slots.size() - 1)]; if (id && id <= frags.size()) __builtin_prefetch(&frags[id - 1]); } }
	void ahead_tail(u64 h) const {
		if (!h || name_slots.empty()) return;
		const u32 id = name_slots[(size_t) h & (name_slots.size() - 1)];
		if (!id || id > frags.size()) return;
		const frag_build& f = frags[id - 1];
		if (f.name_off < names.size()) __builtin_prefetch(names.data() + f.name_off);
		if (f.tail >= 0 && (size_t) f.tail < alns.size()) __builtin_prefetch(&alns[f.tail], 1);
	}
	u32 fragment_lookup(const std::string& name, bool* created, u64 hashed = 0) {
		if (name_slots.empty()) name_slots.assign(1u << 12, 0);
		u64 h = hashed;
		if (!h) { h = 1469598103934665603ULL; for (size_t i = 0; i < name.size(); ++i) { h ^= (u8) name[i]; h *= 1099511628211ULL; } h ^= h >> 29; } // the low bits of the same hash chose the worker
		size_t mask = name_slots.size() - 1, at = (size_t) h & mask;
		for (; name_slots[at] != 0; at = (at + 1) & mask) {
			const frag_build& f = frags[name_slots[at] - 1];
			if (f.name_len == name.size() && memcmp(names.data() + f.name_off, name.data(), name.size()) == 0) { if (created) *created = false; return name_slots[at] - 1; }
		}
		frag_build f; f.name_off = names.size(); f.name_len = (u32) name.size(); f.head = f.tail = -1; f.count = 0; f.single_end = 0; f.duplicate = 0;
		names.insert(names.end(), name.begin(), name.end());
		const u32 id = (u32) frags.size(); frags.push_back(f);
		name_slots[at] = id + 1;
		if (created) *created = true;
		if (frags.size() * 2 > name_slots.size()) resize_name_slots(name_slots.size() * 2); // keep the load below one half
		return id;
	}
	void resize_name_slots(size_t slots) { // a power of two
		std::vector<u32> bigger; bigger.reserve(slots); advise_huge(bigger.data(), slots * sizeof(u32)); bigger.assign(slots, 0); const size_t mask = bigger.size() - 1;
		for (size_t k = 0; k < frags.size(); ++k) {
			const frag_build& g = frags[k];
			u64 hh = 1469598103934665603ULL; for (u32 i = 0; i < g.name_len; ++i) { hh ^= (u8) names[g.name_off + i]; hh *= 1099511628211ULL; }
			hh ^= hh >> 29;
			size_t slot = (size_t) hh & mask; while (bigger[slot] != 0) slot = (slot + 1) & mask;
			bigger[slot] = (u32) k + 1;
		}
		name_slots.swap(bigger);
	}
	// After the first chunk the final size of every pool can be estimated from the share of the file seen so far. Growing a pool by doubling copies it again
	// and again into fresh pages (gigabytes per worker on a large sample); one reservation up front avoids that (it is page-locked and kept for the next sample). A hint only: the
	// pools still grow by themselves where the estimate falls short; `cap_bytes` bounds what one pool may reserve.
	void reserve_ahead(double factor, size_t cap_bytes) {
		auto grow = [&](auto& v) {
			typedef typename std::remove_reference<decltype(v)>::type::value_type value_type;
			const size_t want = std::min((size_t) ((double) v.size() * factor) + 1024, std::max(v.size(), cap_bytes / sizeof(value_type)));
			if (want > v.capacity()) { try { v.reserve(want); advise_huge(v.data(), v.capacity() * sizeof(value_type)); } catch (const std::bad_alloc&) {} } // a hint: no address space, no reservation
		};
		grow(names); grow(cigars); grow(seqs); grow(alns); grow(frags);
		const size_t expected = std::min((size_t) ((double) frags.size() * factor), std::max(frags.size(), cap_bytes / sizeof(frag_build)));
		size_t slots = std::max<size_t>(name_slots.size(), 1u << 12); while (slots < 2 * expected + 16) slots <<= 1;
		if (slots > name_slots.size()) resize_name_slots(slots);
	}
	void link(u32 frag, const aln_build& a) {
		const i32 id = (i32) alns.size(); alns.push_back(a); alns.back().next = -1;
		frag_build& f = frags[frag];
		if (f.tail >= 0) alns[f.tail].next = id; else f.head = id;
		f.tail = id; ++f.count;
	}
	u64 store_seq(const rec_t& r) { // nt16 nibbles copied verbatim, 16-byte aligned
		seqs.resize((seqs.size() + 15) & ~(size_t) 15, 0);
		const u64 off = seqs.size();
		seqs.insert(seqs.end(), r.seq, r.seq + (r.l_seq + 1) / 2);
		return off;
	}
	// converts a BAM record (or a part of it, for read-through alignments) into an alignment of `frag`
	// clip: 0 whole record; 1 keep CIGAR ops from `op` on (clip the start); 2 keep ops up to `op` (clip the end)   (read_chimeric_alignments.cpp:50-91)
	void add_alignment(u32 frag, const rec_t& r, bool supplementary, u32 op = 0, int clip = 0) {
		frag_build& f = frags[frag];
		f.single_end = !(r.flag & BF_PAIRED);
		f.duplicate = f.duplicate || (r.flag & BF_DUP);
		aln_build a; a.supplementary = supplementary; a.first_in_pair = (r.flag & BF_READ1) ? 1 : 0; a.forward = !r.reverse(); a.contig = (u16) r.tid;
		a.seq_off = 0; a.seq_len = 0;
		if (!supplementary) { a.seq_off = store_seq(r); a.seq_len = (u32) r.l_seq; }
		a.cigar_off = (u32) cigars.size();
		if (clip == 1) {
			a.start = r.pos + r.ref_len(op); a.end = r.endpos() - 1;
			const u32 clip_type = (r.cig(0) & 15) == C_H ? C_H : C_S;
			cigars.push_back((u32) r.query_len(op) << 4 | clip_type);
			for (u32 k = op; k < r.n_cigar; ++k) cigars.push_back(r.cig(k));
		} else if (clip == 2) {
			a.start = r.pos; a.end = r.pos + r.ref_len(op + 1) - 1;
			const u32 clip_type = (r.cig(r.n_cigar - 1) & 15) == C_H ? C_H : C_S;
			for (u32 k = 0; k <= op; ++k) cigars.push_back(r.cig(k));
			cigars.push_back((u32) (r.l_seq - r.query_len(op + 1)) << 4 | clip_type);
		} else {
			a.start = r.pos; a.end = r.endpos() - 1;
			for (u32 k = 0; k < r.n_cigar; ++k) cigars.push_back(r.cig(k));
		}
		a.cigar_cnt = (u32) cigars.size() - a.cigar_off;
		link(frag, a);
	}

	// ---- coverage (read_stats.cpp:161-266) ----
	void add_coverage(const rec_t& m1, const rec_t* m2p, bool is_chimeric, bool flags_cleared) {
		const rec_t& m2 = m2p ? *m2p : m1;
		const u16 f1 = flags_cleared ? 0 : m1.flag;
		coverage_windows& cov = *this->cov;
		auto flag = [](u8& x) { __atomic_store_n(&x, (u8) 1, __ATOMIC_RELAXED); };
		if ((u32) m1.tid >= cov.starts.size() || cov.starts[m1.tid].empty() || (u32) m2.tid >= cov.starts.size() || cov.starts[m2.tid].empty()) return;
		if ((f1 & BF_PAIRED) && !(f1 & BF_PROPER)) is_chimeric = true; // the reference's soft-clip tests can never fire (bam_cigar_type() is 0..3)
		if (!is_chimeric) {
			if (!(f1 & BF_REVERSE) || !(f1 & BF_PAIRED)) flag(cov.starts[m1.tid][m1.pos / 20]); else flag(cov.starts[m2.tid][m2.pos / 20]);
		}
		i32 p1 = m1.pos, p2 = m2.pos, position = std::min(p1, p2);
		int window = position / 20;
		u32 i1 = 0, i2 = 0;
		for (;;) {
			u32 c1 = 0, c2 = 0, l1 = 0, l2 = 0;
			if (i1 < m1.n_cigar) { c1 = m1.cig(i1); const u32 o = c1 & 15; l1 = (o == C_M || o == C_D || o == C_N || o == C_EQ || o == C_X) ? c1 >> 4 : 0; } else window = std::max(window, p2 / 20);
			if (i2 < m2.n_cigar) { c2 = m2.cig(i2); const u32 o = c2 & 15; l2 = (o == C_M || o == C_D || o == C_N || o == C_EQ || o == C_X) ? c2 >> 4 : 0; } else window = std::max(window, p1 / 20);
			u32 contig, c;
			if (i1 < m1.n_cigar && (p1 + (i32) l1 < p2 + (i32) l2 || i2 >= m2.n_cigar)) { ++i1; if (l1 == 0) continue; c = c1; contig = (u32) m1.tid; p1 += (i32) l1; position = p1; }
			else if (i2 < m2.n_cigar) { ++i2; if (l2 == 0) continue; c = c2; contig = (u32) m2.tid; p2 += (i32) l2; position = p2; }
			else break;
			const u32 o = c & 15;
			const bool consumes_query = o == C_M || o == C_I || o == C_S || o == C_EQ || o == C_X;
			if (consumes_query) {
				std::vector<u16>& cv = cov.coverage[contig];
				while (window <= position / 20) {
					if (position - window * 20 >= 10) { // saturating increment
						u16 seen = __atomic_load_n(&cv[window], __ATOMIC_RELAXED);
						while (seen < 65535 && !__atomic_compare_exchange_n(&cv[window], &seen, (u16) (seen + 1), true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
					}
					++window;
				}
			} else window = position / 20;
		}
		if (!is_chimeric) {
			if ((f1 & BF_REVERSE) || !(f1 & BF_PAIRED)) flag(cov.ends[m1.tid][(p1 - 1) / 20]); else flag(cov.ends[m2.tid][(p2 - 1) / 20]);
		}
	}

	// ---- internal tandem duplications that the aligner left soft-clipped (read_chimeric_alignments.cpp:197-336) ----
	static bool clipped_sequence_is_adapter(const rec_t& a, const rec_t* bp) {
		if (!bp) return false;
		const rec_t& b = *bp;
		if (a.pos != b.pos) return false;
		const u32 a0 = a.cig(0), al = a.cig(a.n_cigar - 1), b0 = b.cig(0), bl = b.cig(b.n_cigar - 1);
		if (a.reverse() && (a0 & 15) == C_S && !b.reverse() && (bl & 15) == C_S && (a0 >> 4) == (bl >> 4)) return true;
		if (b.reverse() && (b0 & 15) == C_S && !a.reverse() && (al & 15) == C_S && (b0 >> 4) == (al >> 4)) return true;
		return false;
	}
	struct tandem_t { bool forward, first_in_pair, supplementary; u16 contig; i32 start, end; u32 cigar[3]; u32 n_cigar; };
	bool tandem_duplication(const rec_t* rp, tandem_t& t) {
		if (!rp) return false;
		const rec_t& r = *rp;
		const u32 min_clip = 12, min_dup = 9, max_dup = opt->max_itd_length, max_mismatches = 1, max_non_template = 6, min_aligned = 15;
		u32 clip_len = 0, clip_pos = 0; bool clipped_start = true; int direction = +1; int win_start = 0, win_end = 0, ext_start = 0;
		const u32 first = r.cig(0), last = r.cig(r.n_cigar - 1);
		if ((first & 15) == C_S && (first >> 4) >= min_clip) {
			clip_len = first >> 4; clip_pos = 0; direction = -1;
			win_start = (int) ((i64) r.pos + min_dup - clip_len); win_end = (int) ((i64) r.pos + max_dup - clip_len); ext_start = (int) ((i64) r.pos - clip_len); clipped_start = true;
		}
		if ((last & 15) == C_S && (last >> 4) >= std::max(min_clip, clip_len)) {
			clip_len = last >> 4; clip_pos = (u32) r.l_seq - clip_len; direction = +1;
			win_start = (int) ((i64) r.endpos() - max_dup); win_end = (int) ((i64) r.endpos() - min_dup); ext_start = r.endpos(); clipped_start = false;
		}
		if (clip_len == 0) return false;
		if (!ref->has_sequence((u32) r.tid)) return false;
		const char* contig_seq = ref->sequence((u32) r.tid);
		const u64 contig_len = ref->seq_len[r.tid];
		// unsigned comparison on purpose (the reference compares an int sum with a size_t)
		if ((u64) (u32) ((u32) win_end + max_dup + clip_len + 1u) >= contig_len || win_start <= (int) (max_dup + clip_len + 1)) return false;
		// the clipped bases as characters, decoded once: the window scan below compares them ~10^3 times per read
		clip_chars.resize(clip_len);
		for (u32 k = 0; k < clip_len; ++k) clip_chars[k] = nt16_char(r.base_code(clip_pos + k));
		const char* const clip = clip_chars.data();
		// can the read simply be extended linearly? then it is no tandem duplication
		u32 ext_matches = 0;
		for (u32 k = 0; k < clip_len; ++k) {
			const i64 g = (i64) ext_start + k;
			if (g >= 0 && (u64) g < contig_len && contig_seq[g] == clip[k]) ++ext_matches;
		}
		if (1.0 * ext_matches / clip_len >= 0.7f) return false;
		// Quick rejection of a window: the 7th to 14th compared base (positions 6..13 in visiting order) sit in eight consecutive reference bytes. Two
		// mismatches among them end the exact loop below by its 14th step with at most 12 matches -- fewer than min_aligned, and matches + mismatches
		// stays below clip_len when clip_len > 14 -- so such a window cannot be accepted. Random sequence passes this test once in ~2,500 windows.
		const bool prefilter = clip_len > max_non_template + 8 && max_mismatches == 1 && min_aligned > max_non_template + 8 - 2;
		const u32 probe_at = direction == +1 ? max_non_template : clip_len - max_non_template - 8;
		u64 probe = 0; if (prefilter) memcpy(&probe, clip + probe_at, 8);
		for (int cp = win_start; cp <= win_end; ++cp) {
			if (prefilter) {
				u64 refw; memcpy(&refw, contig_seq + cp + probe_at, 8);
				const u64 x = refw ^ probe;
				const u64 nonzero = ((x & 0x7F7F7F7F7F7F7F7FULL) + 0x7F7F7F7F7F7F7F7FULL | x) & 0x8080808080808080ULL; // 0x80 in every byte that differs
				if ((nonzero & (nonzero - 1)) != 0) continue; // at least two bytes differ
			}
			u32 matches = 0, mismatches = 0;
			i64 t_start = (i64) contig_len; i64 t_end = -1;
			for (u32 i = 0; i < clip_len; ++i) {
				const int rp2 = direction == +1 ? (int) i : (int) (clip_len - 1 - i);
				if (contig_seq[cp + rp2] == clip[rp2]) {
					++matches;
					if (cp + rp2 < t_start) t_start = cp + rp2;
					if (cp + rp2 > t_end) t_end = cp + rp2;
				} else if (i >= max_non_template) { if (++mismatches > max_mismatches) break; }
			}
			if (matches >= min_aligned || matches + mismatches == clip_len) {
				t.forward = !r.reverse(); t.first_in_pair = r.flag & BF_READ1; t.contig = (u16) r.tid;
				t.supplementary = !(r.flag & BF_PAIRED) || (clipped_start && !r.reverse()) || (!clipped_start && r.reverse());
				t.start = (i32) t_start; t.end = (i32) t_end;
				u32 clip_left = clipped_start ? 0 : (u32) r.l_seq - clip_len, clip_right = clipped_start ? (u32) r.l_seq - clip_len : 0;
				if (t.start > cp) clip_left += t.start - cp;
				if (t.end < cp + (int) clip_len - 1) clip_right += cp + clip_len - 1 - t.end;
				t.n_cigar = 0;
				if (clip_left > 0) t.cigar[t.n_cigar++] = clip_left << 4 | C_S;
				t.cigar[t.n_cigar++] = (u32) (t.end - t.start + 1) << 4 | C_M;
				if (clip_right > 0) t.cigar[t.n_cigar++] = clip_right << 4 | C_S;
				return true;
			}
		}
		return false;
	}

	// ---- read-through fragments (read_chimeric_alignments.cpp:19-41, 93-193) ----
	static bool spanning_intron(const rec_t& r, i32 gene1_end, i32 gene2_start, u32& op, i32& read_pos) {
		if (r.n_cigar < 3) return false;
		i32 before = r.pos;
		for (u32 k = 0; k < r.n_cigar; ++k) {
			const u32 c = r.cig(k), o = c & 15;
			const i32 len = (o == C_M || o == C_D || o == C_N || o == C_EQ || o == C_X) ? (i32) (c >> 4) : 0;
			const i32 after = before + len;
			if (o == C_N && ((before <= gene1_end && after > gene1_end) || (before < gene2_start && after >= gene2_start))) { op = k; read_pos = r.query_len(k); return true; }
			before = after;
		}
		return false;
	}
	bool extract_read_through(const std::string& name, const rec_t* a, const rec_t* b) {
		const rec_t* fm = a; const rec_t* rm = b;
		if (fm->reverse()) { const rec_t* t = fm; fm = rm; rm = t; }
		idset<1024> fg, rg, common;
		const region_index_view gix = gene_index(an);
		if (fm) query_index(gix, (u32) fm->tid, fm->pos, fm->pos, fg); else query_index(gix, (u32) rm->tid, rm->pos, rm->pos, fg);
		if (rm) query_index(gix, (u32) rm->tid, rm->endpos(), rm->endpos(), rg); else query_index(gix, (u32) fm->tid, fm->endpos(), fm->endpos(), rg);
		if (fg.overflow || rg.overflow) throw std::runtime_error("too many overlapping annotation records at one locus");
		combine_sets(fg.v, fg.n, rg.v, rg.n, common, false);
		if (!(common.n == 0 && !(fg.n == 0 && rg.n == 0))) return false;
		i32 fgs, fge, rgs, rge;
		gene_set_extent(an, fg.v, fg.n, fgs, fge); gene_set_extent(an, rg.v, rg.n, rgs, rge);
		if (fge == -1) fge = rgs - 1;
		if (rgs == -1) rgs = fge + 1;
		u32 fop = 0, rop = 0; i32 fpos = 0, rpos = 0;
		const bool f_intron = fm ? spanning_intron(*fm, fge, rgs, fop, fpos) : false;
		const bool r_intron = rm ? spanning_intron(*rm, fge, rgs, rop, rpos) : false;
		if (f_intron && (!r_intron || fpos < rm->l_seq - rpos)) {
			bool created; const u32 f = fragment(name, &created);
			if (created) {
				add_alignment(f, *fm, false, fop + 1, 1);
				add_alignment(f, *fm, true, fop - 1, 2);
				if (rm) { if (r_intron) add_alignment(f, *rm, false, rop + 1, 1); else add_alignment(f, *rm, false); }
				return true;
			}
		} else if (r_intron) {
			bool created; const u32 f = fragment(name, &created);
			if (created) {
				add_alignment(f, *rm, true, rop + 1, 1);
				add_alignment(f, *rm, false, rop - 1, 2);
				if (fm) { if (f_intron) add_alignment(f, *fm, false, fop - 1, 2); else add_alignment(f, *fm, false); }
				return true;
			}
		} else if (fm && rm && rm->pos >= rgs && fm->endpos() <= fge) {
			bool created; const u32 f = fragment(name, &created);
			if (created) { add_alignment(f, *fm, false); add_alignment(f, *rm, false); }
			return true;
		}
		return false;
	}

	static bool pristine(const rec_t& r) { // read_chimeric_alignments.cpp:526-558
		for (u32 k = 0; k < r.n_cigar; ++k) { const u32 o = r.cig(k) & 15; if (o != C_N && o != C_M && o != C_X) return false; }
		const u32 n = (u32) r.l_seq;
		for (u32 i = 2, repeat = 0, count = 1; i + 2 < n; i += 2) {
			if (r.base_code(i) == r.base_code(repeat) && r.base_code(i + 1) == r.base_code(repeat + 1)) ++count;
			else if (r.base_code(i + 1) == r.base_code(repeat + 1) && r.base_code(i + 2) == r.base_code(repeat + 2)) { ++count; ++i; }
			else { count = 1; repeat = i; }
			if (count >= 8) return false;
		}
		return true;
	}

	// one BAM record, in file order (read_chimeric_alignments.cpp:611-749 for -x input)
	void process(const u8* p, u32 size) {
		rec_t r;
		if (!parse_record(p, size, r)) fail("failed to load alignments");
		++records;
		if ((r.flag & BF_UNMAP) || ((r.flag & BF_PAIRED) && (r.flag & BF_MUNMAP))) return;
		i64 hit_index = 1;
		const u8* hi = find_aux(r, 'H', 'I');
		if (hi) hit_index = aux_int(hi);
		else if (r.flag & BF_SECONDARY) { ++missing_hi; return; }
		key.assign(r.qname, strnlen(r.qname, r.l_qname));
		key += ','; key += std::to_string(hit_index);
		if (r.tid < 0 || (size_t) r.tid >= tid_to_contig->size()) fail("failed to load alignments");
		r.tid = (*tid_to_contig)[r.tid];
		// An alignment that starts before or runs past the end of its contig is not a valid record (SAMv1 1.4), and what the reference does with one is undefined:
		// it indexes its coverage vectors and the contig's sequence beyond their ends (on such a file it aborts in free() or writes garbage columns). Here the same
		// indices would leave the coverage windows on the host and the genome on the device: the run stops with an error instead.
		// Likewise a mapped record without CIGAR operations, or whose CIGAR consumes more bases than the record holds (a sequence of '*' included): the reference
		// dies on those (segmentation fault, or std::out_of_range from substr); everything downstream indexes the sequence by the CIGAR.
		i64 ref_span = 0, query_span = 0;
		for (u32 k = 0; k < r.n_cigar; ++k) { const u32 c = r.cig(k), o = c & 15; if (o == C_M || o == C_EQ || o == C_X) { ref_span += c >> 4; query_span += c >> 4; } else if (o == C_D || o == C_N) ref_span += c >> 4; else if (o == C_I || o == C_S) query_span += c >> 4; }
		if (r.n_cigar == 0 || query_span > (i64) r.l_seq)
			fail("CIGAR string of read '" + std::string(r.qname, strnlen(r.qname, r.l_qname)) + "' does not fit its sequence (" + std::to_string(query_span) + " bases in " + std::to_string(r.n_cigar) + " operations, sequence of " + std::to_string(r.l_seq) + ")");
		if (ref->has_sequence((u32) r.tid) && (r.pos < 0 || (i64) r.pos + (ref_span ? ref_span : 1) > (i64) ref->seq_len[r.tid]))
			fail("alignment of read '" + std::string(r.qname, strnlen(r.qname, r.l_qname)) + "' extends beyond the end of contig '" + ref->original_names[r.tid] + "' (was the file aligned to another assembly?)");

		if (r.flag & BF_SUPPLEMENTARY) {
			if (clipped_at_correct_end(r)) add_alignment(fragment(key, NULL, key_hash_hint), r, true); else ++malformed;
			no_chimeric = false;
			return;
		}
		if ((*interesting_contig)[r.tid]) ++mapped_reads;
		if ((r.flag & BF_PAIRED) && !(r.flag & BF_PROPER)) { // discordant mate
			add_alignment(fragment(key, NULL, key_hash_hint), r, false);
			no_chimeric = false;
			if (!opt->external_duplicate_marking || !(r.flag & BF_DUP)) add_coverage(r, NULL, true, true); // all flag bits cleared (`flag &= !BAM_FPAIRED`)
			return;
		}
		rec_t mate; mate.base = NULL;
		std::vector<u8> mate_bytes;
		if (r.flag & BF_PAIRED) {
			// The first mate of a proper pair waits for the second. Mates are neighbours in a collated BAM: the most recent waiting record is only
			// remembered by its address in the chunk buffer and moves into the map (a copy) when another name arrives or the chunk ends.
			if (waiting_ptr && waiting_key == key) {
				parse_record(waiting_ptr, waiting_size, mate); waiting_ptr = NULL;
			} else {
				std::unordered_map<std::string, std::vector<u8>, name_hash>::iterator it = pending.find(key);
				if (it == pending.end()) { park_waiting(); waiting_ptr = p; waiting_size = size; waiting_key = key; return; }
				mate_bytes.swap(it->second); pending.erase(it);
				parse_record(mate_bytes.data(), (u32) mate_bytes.size(), mate);
			}
			mate.tid = (*tid_to_contig)[mate.tid];
		}
		const rec_t* m = mate.valid() ? &mate : NULL;
		bool is_tandem = false;
		tandem_t t;
		bool tandem_from_record = false, tandem_from_mate = false;
		if (!clipped_sequence_is_adapter(r, m) && (!m || r.reverse() != m->reverse())) {
			tandem_from_record = tandem_duplication(&r, t);
			if (!tandem_from_record) tandem_from_mate = tandem_duplication(m, t);
		}
		if (tandem_from_record || tandem_from_mate) {
			const u32 f = fragment(key + "ITD");
			add_alignment(f, r, (!r.reverse()) == t.forward && !t.supplementary);
			if (m) add_alignment(f, *m, (!m->reverse()) == t.forward && !t.supplementary);
			aln_build a; a.supplementary = t.supplementary; a.first_in_pair = t.first_in_pair; a.forward = t.forward; a.contig = t.contig; a.start = t.start; a.end = t.end;
			a.seq_off = 0; a.seq_len = 0;
			if (!t.supplementary) { const rec_t& src = tandem_from_mate ? *m : r; a.seq_off = store_seq(src); a.seq_len = (u32) src.l_seq; }
			a.cigar_off = (u32) cigars.size(); for (u32 k = 0; k < t.n_cigar; ++k) cigars.push_back(t.cigar[k]); a.cigar_cnt = t.n_cigar;
			link(f, a);
			is_tandem = true;
		}
		bool is_read_through = false;
		if ((find_aux(r, 'S', 'A') && clipped_at_correct_end(r)) || (m && find_aux(*m, 'S', 'A') && clipped_at_correct_end(*m))) {
			const u32 f = fragment(key, NULL, key_hash_hint);
			add_alignment(f, r, false);
			if (m) add_alignment(f, *m, false);
			no_chimeric = false;
		} else if (!is_tandem) {
			is_read_through = extract_read_through(key, &r, m);
			if ((*viral_contig)[r.tid]) {
				if (pristine(r)) ++viral_reads[r.tid];
				if (m && pristine(*m)) ++viral_reads[m->tid];
			}
		}
		if (!opt->external_duplicate_marking || !(r.flag & BF_DUP)) add_coverage(r, m, is_read_through, false);
	}
};


// workers of finished samples, kept for the next one (one set; a set is only reused by a run with the same number of workers)
static std::mutex g_worker_cache_lock; static std::vector<worker>* g_worker_cache = NULL;
static std::vector<worker>* take_workers(int T) {
	std::vector<worker>* set = NULL;
	{ std::lock_guard<std::mutex> g(g_worker_cache_lock); set = g_worker_cache; g_worker_cache = NULL; }
	if (set && (int) set->size() != T) { std::thread([set]() { delete set; }).detach(); set = NULL; } // unmapping gigabytes takes most of a second: not on this thread
	return set ? set : new std::vector<worker>(T);
}
static void put_workers(std::vector<worker>* set) { // recycled by a helper thread: clearing the name slots touches every page of them once
	std::thread([set]() {
		for (size_t t = 0; t < set->size(); ++t) (*set)[t].recycle();
		std::vector<worker>* old = NULL;
		{ std::lock_guard<std::mutex> g(g_worker_cache_lock); old = g_worker_cache; g_worker_cache = set; }
		delete old;
	}).detach();
}
void release_worker_cache() { std::vector<worker>* old = NULL; { std::lock_guard<std::mutex> g(g_worker_cache_lock); old = g_worker_cache; g_worker_cache = NULL; } delete old; }

// ------------------------------------------------------------------------------------------- BGZF container
struct bgzf_file {
	const u8* data; size_t size; int fd;
	struct block { u64 in_off; u32 in_len; u32 out_len; u64 out_off; };
	std::vector<block> blocks; u64 total_out;
	bgzf_file(): data(NULL), size(0), fd(-1), total_out(0) {}
	~bgzf_file() { if (data) munmap((void*) data, size); if (fd >= 0) close(fd); }
	void open(const std::string& path, int threads) {
		fd = ::open(path.c_str(), O_RDONLY);
		if (fd < 0) fail("failed to open SAM file");
		struct stat st; fstat(fd, &st); size = st.st_size;
		if (size == 0) fail("failed to read SAM header");
		data = (const u8*) mmap(NULL, size, PROT_READ, MAP_PRIVATE, fd, 0);
		if (data == MAP_FAILED) { data = NULL; fail("failed to open SAM file"); }
		madvise((void*) data, size, MADV_SEQUENTIAL);
		// Block table. A block is found from the one before it (its size sits in its header), and every header read faults a page of the mapping in: a
		// 7 GB file of stored blocks costs a quarter of a second on one thread. So every piece of the file guesses its first block (two well-formed
		// headers in a row), walks from there, and the guesses are VERIFIED: the chain of piece s must arrive exactly at the guess of piece s+1; where it
		// does not, that stretch is walked serially. Errors are raised by the serial walk only, at the same offsets as before.
		auto header = [&](u64 off, u32& bsize, u32& xlen) { // well-formed BGZF header at off (SAMv1 4.1)?
			if (off + 18 > size) return false;
			const u8* h = data + off;
			if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) return false;
			xlen = rd16(h + 10);
			if (off + 12 + xlen > size) return false;
			bool found = false;
			for (u32 x = 0; x + 4 <= xlen;) { const u8* e = h + 12 + x; const u32 slen = rd16(e + 2); if (e[0] == 'B' && e[1] == 'C' && slen == 2) { bsize = rd16(e + 4) + 1u; found = true; } x += 4 + slen; }
			return found && bsize >= 12 + xlen + 8 && off + bsize <= size;
		};
		auto walk = [&](u64 off, u64 limit, std::vector<block>& out, bool strict) { // blocks starting before `limit`; returns where the chain stands
			while (off < limit && off + 18 <= size) {
				u32 bsize = 0, xlen = 0;
				if (!header(off, bsize, xlen)) {
					if (!strict) break;
					const u8* h = data + off;
					const bool magic = h[0] == 0x1f && h[1] == 0x8b && h[2] == 8 && (h[3] & 4);
					fail(!magic && off == 0 ? "failed to read SAM header" : "failed to load alignments"); // not BGZF (SAM text / CRAM are not supported); at the start of the file no header can be read (arriba.cpp:122)
				}
				block b; b.in_off = off + 12 + xlen; b.in_len = bsize - 12 - xlen - 8; b.out_len = rd32(data + off + bsize - 4); b.out_off = 0;
				out.push_back(b);
				off += bsize;
			}
			return off;
		};
		const size_t min_bytes = getenv("ARB_SCAN_MIN_BYTES") ? (size_t) atol(getenv("ARB_SCAN_MIN_BYTES")) : (size_t) 64 << 20; // test hook
		const int pieces = threads > 1 && size > min_bytes ? threads : 1;
		if (pieces > 1) {
			std::vector<u64> guess(pieces + 1, size), stop_at(pieces, 0);
			std::vector<std::vector<block> > found(pieces);
			guess[0] = 0;
			std::vector<std::thread> pool;
			for (int s = 1; s < pieces; ++s) pool.emplace_back([&, s]() {
				u64 q = (u64) size * s / pieces; const u64 give_up = std::min<u64>(size, q + (256u << 10));
				for (; q < give_up; ++q) { u32 b1 = 0, x1 = 0, b2 = 0, x2 = 0; if (header(q, b1, x1) && (q + b1 + 18 > size || header(q + b1, b2, x2))) break; }
				guess[s] = q < give_up ? q : size;
			});
			for (size_t t = 0; t < pool.size(); ++t) pool[t].join();
			pool.clear();
			for (int s = 1; s < pieces; ++s) pool.emplace_back([&, s]() { stop_at[s] = guess[s] < size ? walk(guess[s], guess[s + 1], found[s], false) : size; });
			stop_at[0] = walk(0, guess[1], found[0], false);
			for (size_t t = 0; t < pool.size(); ++t) pool[t].join();
			u64 q = 0;
			for (int s = 0; s < pieces; ++s) {
				if (q == guess[s] && guess[s] < size) { blocks.insert(blocks.end(), found[s].begin(), found[s].end()); q = stop_at[s]; }
				if (q < guess[s + 1]) q = walk(q, guess[s + 1], blocks, true); // wrong or missing guess, or a chain that broke off: walk (and diagnose) this stretch
			}
			walk(q, size, blocks, true);
		} else walk(0, size, blocks, true);
		u64 out = 0;
		for (size_t b = 0; b < blocks.size(); ++b) { blocks[b].out_off = out; out += blocks[b].out_len; }
		total_out = out;
	}
	void inflate_block(const block& b, u8* dst) const {
		if (b.out_len == 0) return;
		// STAR is run with --outBAMcompression 0 (run_arriba.sh:34): every BGZF block then holds ONE stored deflate block -- header byte 0x01 (final, type 00),
		// LEN, ~LEN, the bytes (RFC 1951 3.2.4). Those are copied; anything else goes through zlib.
		const u8* const in = data + b.in_off;
		if (b.in_len == 5ull + b.out_len && in[0] == 0x01 && rd16(in + 1) == (u16) b.out_len && (u16) (rd16(in + 1) ^ rd16(in + 3)) == 0xFFFF) { memcpy(dst, in + 5, b.out_len); return; }
		z_stream zs; memset(&zs, 0, sizeof(zs));
		if (inflateInit2(&zs, -15) != Z_OK) fail("failed to load alignments");
		zs.next_in = (Bytef*) (data + b.in_off); zs.avail_in = b.in_len; zs.next_out = dst; zs.avail_out = b.out_len;
		const int rc = inflate(&zs, Z_FINISH);
		inflateEnd(&zs);
		if (rc != Z_STREAM_END || zs.avail_out != 0) fail("failed to load alignments");
	}
};

template <class F> static void parallel_for(int threads, size_t n, F f) { // f(thread, begin, end)
	if (threads <= 1 || n < 2) { f(0, (size_t) 0, n); return; }
	std::vector<std::thread> pool; std::vector<std::string> errors(threads);
	for (int t = 0; t < threads; ++t) pool.emplace_back([&, t]() {
		try { f(t, n * t / threads, n * (t + 1) / threads); } catch (const std::exception& e) { errors[t] = e.what(); }
	});
	for (size_t t = 0; t < pool.size(); ++t) pool[t].join();
	for (int t = 0; t < threads; ++t) if (!errors[t].empty()) fail(errors[t]);
}

// ------------------------------------------------------------------------------------------- driver
frag_view fragment_table::view() {
	frag_view v;
	v.n = n; v.n_aln = n_aln.data(); v.fflags = fflags.data(); v.filter = filter.data(); v.contig = contig.data(); v.start = start.data(); v.end = end.data();
	v.aflags = aflags.data(); v.cigar_off = cigar_off.data(); v.cigar_cnt = cigar_cnt.data(); v.seq_off = seq_off.data(); v.seq_len = seq_len.data();
	v.genes_off = genes_off.data(); v.genes_cnt = genes_cnt.data(); v.cigar = cigar.data(); v.seq = seq.data(); v.genes = genes.data();
	return v;
}


void read_chimeric_alignments(const std::string& bam_path, refdata& ref, const ingest_options& opt, fragment_table& out, coverage_windows& coverage, ingest_stats& stats) {
	const int T = std::min(255, std::max(1, opt.threads)); // shard ids are bytes
	double t0 = now_s();
	const bool trace = getenv("ARB_TRACE") != NULL;
	double tr_last = t0;
	auto lap = [&](const char* what) { if (trace) { const double t = now_s(); fprintf(stderr, "[ingest] %-28s %.3f s\n", what, t - tr_last); tr_last = t; } };
	bgzf_file bam; bam.open(bam_path, T);
	lap("open + block table");
	stats.t_inflate = stats.t_parse = stats.t_finalize = 0;

	// chunks of ~128 MiB of decompressed data, each a whole number of BGZF blocks; a record that straddles a chunk
	// boundary is carried over to the front of the next buffer
	const u64 chunk_target = getenv("ARB_CHUNK_BYTES") ? (u64) atoll(getenv("ARB_CHUNK_BYTES")) : 128ull << 20; // env: test hook (many small chunks)
	struct worker_set { std::vector<worker>* set; explicit worker_set(int n): set(take_workers(n)) {} ~worker_set() { if (set) put_workers(set); } } held(T); // back to the cache on every way out
	std::vector<worker>& workers = *held.set;
	std::vector<u16> tid_to_contig; std::vector<u8> interesting_contig, viral_contig;
	bool header_done = false;
	u64 total_records = 0;
	// A chunk is inflated, cut into records and sharded ("prepare") while the workers still parse the previous one ("process").
	struct chunk_t { column<u8> buf /* page-locked: copied to the device for the record scan */; column<u32> shard_rec_off /* record offsets, worker by worker, file order inside a worker's list */; std::vector<u32> shard_begin; size_t n_records, consumed; bool last; chunk_t(): n_records(0), consumed(0), last(false) {} };
	chunk_t chunks[2];
	size_t b0 = 0;
	double t_inflate = 0, t_scan = 0; // written by the preparing thread only
	auto prepare = [&](chunk_t& c, const chunk_t* prev) {
		const size_t carry = prev ? prev->buf.size() - prev->consumed : 0;
		size_t b1 = b0; u64 bytes = 0;
		while (b1 < bam.blocks.size() && (bytes == 0 || bytes + bam.blocks[b1].out_len <= chunk_target)) bytes += bam.blocks[b1++].out_len;
		if (b1 == b0 && carry > 0) fail("failed to load alignments"); // truncated file
		column<u8>& buf = c.buf;
		if (buf.capacity() < carry + bytes) buf.reserve(carry + bytes + (16u << 20)); // one page-locked block per buffer for the whole file (chunks differ a little in size)
		buf.resize(carry + bytes);
		if (carry) memcpy(buf.data(), prev->buf.data() + prev->consumed, carry);
		double ti = now_s();
		const u64 base_out = b0 < bam.blocks.size() ? bam.blocks[b0].out_off : 0;
		const size_t first = b0;
		parallel_for(T, b1 - first, [&](int, size_t lo, size_t hi) { for (size_t b = first + lo; b < first + hi; ++b) bam.inflate_block(bam.blocks[b], buf.data() + carry + (bam.blocks[b].out_off - base_out)); });
		t_inflate += now_s() - ti;
		b0 = b1;
		c.last = b0 >= bam.blocks.size();
		size_t p = 0;
		if (!header_done) {
			if (buf.size() < 12 || memcmp(buf.data(), "BAM\1", 4) != 0) fail("failed to read SAM header");
			const u32 l_text = rd32(buf.data() + 4);
			if (12ull + l_text > buf.size()) fail("failed to read SAM header (header larger than one chunk)");
			p = 8 + l_text;
			const u32 n_ref = rd32(buf.data() + p); p += 4;
			tid_to_contig.resize(n_ref);
			for (u32 k = 0; k < n_ref; ++k) {
				if (p + 4 > buf.size()) fail("failed to read SAM header");
				const u32 l_name = rd32(buf.data() + p); p += 4;
				if (p + l_name + 4 > buf.size()) fail("failed to read SAM header");
				const std::string target((const char*) buf.data() + p, strnlen((const char*) buf.data() + p, l_name)); p += l_name + 4;
				const std::string name = remove_chr(target);
				const u16 id = ref.contig_id(name);
				ref.original_names[id] = target;
				tid_to_contig[k] = id;
			}
			const size_t nc = ref.contig_ids.size();
			interesting_contig.assign(nc, 0); viral_contig.assign(nc, 0);
			for (std::map<std::string, u16>::iterator c = ref.contig_ids.begin(); c != ref.contig_ids.end(); ++c) {
				interesting_contig[c->second] = contig_matches(c->first, opt.interesting_contigs);
				viral_contig[c->second] = contig_matches(c->first, opt.viral_contigs);
				if (!ref.has_sequence(c->second) && interesting_contig[c->second]) fail("could not find sequence of contig '" + c->first + "'");
			}
			ref.flatten(); // contig table may have grown
			coverage.resize(ref);
			for (int t = 0; t < T; ++t) {
				worker& w = workers[t];
				w.ref = &ref; w.opt = &opt; w.tid_to_contig = &tid_to_contig; w.interesting_contig = &interesting_contig; w.viral_contig = &viral_contig;
				w.an = ref.host_view(); w.viral_reads.assign(nc, 0);
				w.cov = &coverage;
			}
			header_done = true;
		}
		// record boundaries, read-name hashes and the per-worker record lists: on the device (csrc/bamscan.cu)
		double tp = now_s();
		{
			if (buf.size() >= 0xFFFFFFF0ull) fail("failed to load alignments (chunk too large)");
			c.shard_begin.assign((size_t) T + 1, 0);
			c.shard_rec_off.resize(buf.size() / 36 + 2);
			uint64_t consumed = 0; uint32_t n_records = 0, malformed = 0;
			if (arb_bam_scan(opt.scan_ctx, buf.data(), buf.size(), p, (int32_t) tid_to_contig.size(), (uint32_t) T, &consumed, &n_records, c.shard_begin.data(), c.shard_rec_off.data(), &malformed) != 0)
				fail(std::string("arb_bam_scan: ") + arb_last_error(opt.scan_ctx));
			if (malformed) fail("failed to load alignments");
			c.n_records = n_records; p = consumed;
		}
		c.consumed = p;
		t_scan += now_s() - tp;
		if (c.last && c.consumed != buf.size()) fail("failed to load alignments");
	};
	if (bam.blocks.empty()) fail("failed to read SAM header");
	prepare(chunks[0], NULL);
	bool reserved_ahead = false;
	const bool look_ahead = getenv("ARB_INGEST_LOOKAHEAD") == NULL || atoi(getenv("ARB_INGEST_LOOKAHEAD")) != 0;
	for (int cur = 0;; cur ^= 1) {
		chunk_t& c = chunks[cur];
		std::string prepare_error; std::thread next;
		if (!c.last) next = std::thread([&]() { try { prepare(chunks[cur ^ 1], &c); } catch (const std::exception& x) { prepare_error = x.what(); if (prepare_error.empty()) prepare_error = "failed to load alignments"; } });
		const double tp = now_s();
		std::string process_error;
		try {
			total_records += c.n_records;
			parallel_for(T, (size_t) T, [&](int, size_t lo, size_t hi) {
				for (size_t t = lo; t < hi; ++t) {
					worker& w = workers[t];
					const u8* base = c.buf.data();
					const u32* const mine = c.shard_rec_off.data(); const u32 stop = c.shard_begin[t + 1];
					u64 ring[8] = {0, 0, 0, 0, 0, 0, 0, 0}; // key hashes of the records ahead (worker::ahead_hash)
					const u32 first = c.shard_begin[t];
					for (u32 x = first; x < stop; ++x) {
						if (look_ahead) {
							if (x + 9 < stop) { const u8* ahead = base + mine[x + 9]; __builtin_prefetch(ahead); __builtin_prefetch(ahead + 64); __builtin_prefetch(ahead + 192); __builtin_prefetch(ahead + 256); } // fixed fields + name, and where the tags of a 2x101 / 2x151 record start
							if (x == first) for (u32 y = x; y < x + 5 && y < stop; ++y) ring[y & 7] = w.ahead_hash(base + mine[y] + 4, rd32(base + mine[y]));
							if (x + 5 < stop) ring[(x + 5) & 7] = w.ahead_hash(base + mine[x + 5] + 4, rd32(base + mine[x + 5]));
							if (x + 3 < stop) w.ahead_fragment(ring[(x + 3) & 7]);
							if (x + 1 < stop) w.ahead_tail(ring[(x + 1) & 7]);
							w.key_hash_hint = ring[x & 7];
						} else if (x + 3 < stop) { const u8* ahead = base + mine[x + 3]; __builtin_prefetch(ahead); __builtin_prefetch(ahead + 64); __builtin_prefetch(ahead + 192); __builtin_prefetch(ahead + 256); }
						const u64 off = mine[x];
						w.process(base + off + 4, rd32(base + off));
					}
					w.key_hash_hint = 0;
					w.park_waiting();
				}
			});
		} catch (const std::exception& x) { process_error = x.what(); }
		stats.t_parse += now_s() - tp;
		if (cur == 0 && !reserved_ahead && !c.last && process_error.empty() && c.consumed > 0) { // once, after the first chunk
			reserved_ahead = true;
			const double factor = 1.03 * (double) bam.total_out / (double) c.consumed;
			parallel_for(T, (size_t) T, [&](int, size_t lo, size_t hi) { for (size_t t = lo; t < hi; ++t) workers[t].reserve_ahead(factor, (size_t) (1.5 * (double) bam.total_out / T)); });
		}
		if (next.joinable()) next.join();
		if (!process_error.empty()) fail(process_error);
		if (!prepare_error.empty()) fail(prepare_error);
		if (c.last) break;
	}
	if (trace) fprintf(stderr, "[ingest]   of which inflate %.3f s, record scan + name hashing %.3f s (both overlap with) record processing %.3f s\n", t_inflate, t_scan, stats.t_parse);
	stats.t_inflate = t_inflate; stats.t_parse += t_scan;
	{ chunk_t a, b; std::swap(chunks[0], a); std::swap(chunks[1], b); }
	if (!header_done) fail("failed to read SAM header");
	(void) t0;
	lap("inflate + scan + parse");

	// ---- merge by-products ----
	double tf = now_s();
	stats.mapped_reads = 0; stats.malformed = 0; stats.missing_hi_tag = 0; stats.records = total_records; stats.no_chimeric_reads = true;
	stats.mapped_viral_reads_by_contig.assign(ref.contig_ids.size(), 0);
	for (int t = 0; t < T; ++t) {
		worker& w = workers[t];
		stats.mapped_reads += w.mapped_reads; stats.malformed += w.malformed; stats.missing_hi_tag += w.missing_hi; stats.no_chimeric_reads = stats.no_chimeric_reads && w.no_chimeric;
		for (size_t c = 0; c < w.viral_reads.size(); ++c) stats.mapped_viral_reads_by_contig[c] += w.viral_reads[c];
	}
	lap("merge by-products");
	if (stats.mapped_reads == 0) fail("no normal reads found");

	// ---- the fragment table: slot normalisation, name order, columns and multimapper flags, on the device (csrc/fragtable.cu) ----
	std::vector<arb_ingest_pool> pools(T);
	for (int t = 0; t < T; ++t) {
		const worker& w = workers[t]; arb_ingest_pool& q = pools[t];
		q.names = w.names.data(); q.n_name_bytes = w.names.size(); q.cigars = w.cigars.data(); q.n_cigars = w.cigars.size(); q.seqs = w.seqs.data(); q.n_seq_bytes = w.seqs.size();
		q.alns = w.alns.data(); q.n_alns = w.alns.size(); q.frags = w.frags.data(); q.n_frags = (u32) w.frags.size();
	}
	arb_fragment_table_sizes sz;
	if (arb_build_fragment_table(opt.scan_ctx, pools.data(), (u32) T, &sz) != 0) fail(arb_last_error(opt.scan_ctx));
	if (trace) fprintf(stderr, "[ingest]   of which pools -> device %.1f ms, whole device build %.1f ms, %u name-sort rounds past the first 16 bytes\n", sz.upload_ms, sz.build_ms, sz.tie_rounds);
	lap("fragment table (device)");
	stats.malformed += sz.n_rejected;
	if (stats.malformed > 0) std::cerr << "WARNING: " << stats.malformed << " SAM records were malformed and ignored" << std::endl;
	if (stats.no_chimeric_reads) fail("no split reads or discordant mates found (STAR must either be run with '--chimOutType WithinBAM' or the file 'Chimeric.out.sam' must be passed to Arriba via the argument -c)");
	if (stats.missing_hi_tag > 0) std::cerr << "WARNING: " << stats.missing_hi_tag << " secondary alignments lack the 'HI' tag and were ignored (STAR must be run with '--outSAMattributes HI' for Arriba to make use of multi-mapping reads for fusion detection)" << std::endl;

	// ---- the host image of the table (strandedness, fragment length, the event glue and the output read it) ----
	const u32 n = sz.n_fragments;
	const size_t n3 = 3 * (size_t) n;
	out.n = n;
	out.n_aln.resize(n); out.fflags.resize(n); out.filter.resize(n);
	out.contig.resize(n3); out.start.resize(n3); out.end.resize(n3); out.aflags.resize(n3); out.cigar_off.resize(n3); out.cigar_cnt.resize(n3);
	out.seq_off.resize(2 * (size_t) n); out.seq_len.resize(2 * (size_t) n); out.genes_off.resize(n3); out.genes_cnt.resize(n3);
	out.cigar.resize(sz.n_cigar); out.seq.resize(sz.n_seq_bytes); out.names.resize(sz.n_name_bytes); out.name_off.resize((size_t) n + 1);
	// the gene sets come with the annotation; until then they are empty (zeroed here while the copies run)
	std::thread zero_genes([&]() { memset(out.genes_off.data(), 0, n3 * sizeof(u32)); memset(out.genes_cnt.data(), 0, n3 * sizeof(u16)); });
	arb_fragment_columns cols = {out.n_aln.data(), out.fflags.data(), out.filter.data(), out.contig.data(), out.start.data(), out.end.data(), out.aflags.data(), out.cigar_off.data(),
	                             out.cigar_cnt.data(), out.seq_off.data(), out.seq_len.data(), out.cigar.data(), out.seq.data(), out.names.data(), out.name_off.data()};
	const int rc = arb_get_fragment_table(opt.scan_ctx, &cols);
	zero_genes.join();
	if (rc != 0) fail(arb_last_error(opt.scan_ctx));
	stats.t_finalize = now_s() - tf;
	lap("fragment table -> host");
	// the workers go back to the cache when `held` leaves scope (their contents are dropped by a helper thread)
	lap("free worker state");
}

}} // namespace
