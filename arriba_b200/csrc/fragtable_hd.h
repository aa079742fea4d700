// fragtable_hd.h -- rules of the fragment table that ingest hands to the later stages: slot normalisation and rejection of malformed fragments
// (read_chimeric_alignments.cpp:340-373 disjoin_split_read_segments, :377-506 remove_malformed_alignments), the name order of the fragments (the std::map
// order of "<qname>,<HI>[ITD]") and the multimapper flags (mark_multimappers, :792-802). The driver is fragtable.cu.
#pragma once
#include "prims.h"
#include "model.h"
#include "../../include/arriba_b200.h"

namespace arb {

// The workers' pools, concatenated worker after worker on the device. A fragment's id is its worker's base + its id in the worker; every offset inside
// a pool record is relative to that worker's stretch of the pool.
struct pool_view {
	const char* names; const u32* cigars; const u8* seqs; const arb_pool_alignment* alns; const arb_pool_fragment* frags;
	const u64* name_base; const u64* cigar_base; const u64* seq_base; const u64* aln_base; const u32* frag_base; u32 n_workers;
	ARB_HD u32 worker_of(u32 g) const { // last worker whose first fragment is <= g (workers without fragments share their base with the next one)
		u32 lo = 0, hi = n_workers; // frag_base[lo] <= g < frag_base[hi]
		while (hi - lo > 1) { const u32 mid = (lo + hi) / 2; if (frag_base[mid] <= g) lo = mid; else hi = mid; }
		return lo;
	}
	ARB_HD const char* name(u32 g, u32& len) const { const u32 w = worker_of(g); const arb_pool_fragment& f = frags[g]; len = f.name_len; return names + name_base[w] + f.name_off; }
	// bytes 8w .. 8w+7 of a name as a big-endian word, zero bytes past its end: names hold no NUL, so comparing these words word by word is
	// std::string::compare (a name that is a prefix of another one sorts first)
	ARB_HD u64 name_word(u32 g, u32 w) const {
		u32 len; const char* s = name(g, len);
		u64 v = 0;
		for (u32 k = 0; k < 8; ++k) { const u32 at = 8 * w + k; v = v << 8 | (at < len ? (u64) (u8) s[at] : 0); }
		return v;
	}
};

// One alignment during normalisation: its pool record, its CIGAR in the pool and the operations normalisation rewrote. Normalisation never changes how
// many operations an alignment has and edits at most two of them (a clip at either end, or the clip and the match next to it), so the CIGAR stays in the pool.
struct norm_slot {
	arb_pool_alignment a; const u32* cig; u32 cnt; u32 n_edits; u32 edit_at[4], edit_to[4];
	ARB_HD u32 op(u32 k) const { for (u32 e = n_edits; e-- > 0;) if (edit_at[e] == k) return edit_to[e]; return cig[k]; }
	ARB_HD void set(u32 k, u32 v) { for (u32 e = 0; e < n_edits; ++e) if (edit_at[e] == k) { edit_to[e] = v; return; } edit_at[n_edits] = k; edit_to[n_edits] = v; ++n_edits; }
	ARB_HD u32 front() const { return op(0); }
	ARB_HD u32 back() const { return op(cnt - 1); }
	ARB_HD u32 clip(bool at_front) const { const u32 c = at_front ? front() : back(); return cig_is_clip(c) ? c >> 4 : 0; }
};
ARB_HD void swap_slots(norm_slot& x, norm_slot& y) { norm_slot t = x; x = y; y = t; }

ARB_HD bool disjoin_segments(norm_slot& split, norm_slot& supp) {
	const u32 clipped_split = split.a.forward ? split.clip(true) : split.clip(false);
	const u32 clipped_supp = supp.a.forward ? supp.clip(false) : supp.clip(true);
	const int overlap = (int) split.a.seq_len - (int) clipped_split - (int) clipped_supp;
	if (overlap <= 0) return true;
	const u32 clipped_op = supp.a.forward ? supp.cnt - 1 : 0;
	const u32 matching_op = supp.a.forward ? clipped_op - 1 : 1;
	if (supp.cnt < 2 || (supp.op(matching_op) & 15) != C_M || (int) (supp.op(matching_op) >> 4) < overlap + 10) return false;
	const u32 c = supp.op(clipped_op), m = supp.op(matching_op);
	supp.set(clipped_op, ((c >> 4) + overlap) << 4 | (c & 15));
	supp.set(matching_op, ((m >> 4) - overlap) << 4 | (m & 15));
	if (supp.a.forward) supp.a.end -= overlap; else supp.a.start += overlap;
	return true;
}

// Brings a fragment's alignments (m[0..n), in the order they were linked) into the canonical slots MATE1, MATE2 / SPLIT_READ, SUPPLEMENTARY, or rejects it.
ARB_HD bool normalise_fragment(norm_slot* m, u32& n, bool single_end) {
	if (single_end) {
		if (!(n == 2 && (m[0].a.supplementary != m[1].a.supplementary))) return false;
		// the longer anchor becomes the split read; it is duplicated into the MATE1 slot to imitate paired-end data
		if (m[0].a.end - m[0].a.start > m[1].a.end - m[1].a.start) { m[2] = m[1]; m[1] = m[0]; }
		else { m[2] = m[0]; m[0] = m[1]; }
		n = 3;
		// sequence: MATE1 and SPLIT_READ carry it, SUPPLEMENTARY does not
		if (!m[0].a.supplementary) { m[1].a.seq_off = m[0].a.seq_off; m[1].a.seq_len = m[0].a.seq_len; }
		else if (!m[1].a.supplementary) { m[0].a.seq_off = m[1].a.seq_off; m[0].a.seq_len = m[1].a.seq_len; }
		else { m[0].a.seq_off = m[1].a.seq_off = m[2].a.seq_off; m[0].a.seq_len = m[1].a.seq_len = m[2].a.seq_len; }
		m[2].a.seq_len = 0;
		for (int s = 0; s < 2; ++s) {
			if ((m[s].front() & 15) == C_H) m[s].set(0, (m[s].front() >> 4) << 4 | C_S);
			if ((m[s].back() & 15) == C_H) {
				// the reference takes the length for SPLIT_READ's last op from MATE1's CIGAR at the same index (read_chimeric_alignments.cpp:415)
				const u32 len = s == 0 ? m[0].back() >> 4 : (m[1].cnt - 1 < m[0].cnt ? m[0].op(m[1].cnt - 1) >> 4 : 0);
				m[s].set(m[s].cnt - 1, len << 4 | C_S);
			}
		}
		m[2].a.supplementary = 1; m[0].a.supplementary = 0; m[1].a.supplementary = 0;
		const bool same = m[1].a.forward == m[2].a.forward;
		const u32 len = m[1].a.seq_len;
		const u32 lhs = len - m[1].clip(true) - (same ? m[2].clip(false) : m[2].clip(true));
		const u32 rhs = len - m[1].clip(false) - (same ? m[2].clip(true) : m[2].clip(false));
		const bool flip = lhs < rhs ? (m[1].a.forward != 0) : (m[1].a.forward == 0);
		if (flip) m[0].a.forward = !m[0].a.forward; else { m[1].a.forward = !m[1].a.forward; m[2].a.forward = !m[2].a.forward; }
		m[0].a.first_in_pair = !flip; m[1].a.first_in_pair = flip; m[2].a.first_in_pair = flip;
		if (!disjoin_segments(m[1], m[2])) return false;
	} else if (n == 3) {
		if (m[0].a.supplementary) swap_slots(m[0], m[2]); else if (m[1].a.supplementary) swap_slots(m[1], m[2]);
		if (m[1].a.first_in_pair != m[2].a.first_in_pair) swap_slots(m[0], m[1]);
		if (m[0].a.supplementary || m[1].a.supplementary || !m[2].a.supplementary) return false;
		if (m[0].a.contig != m[1].a.contig || m[0].a.forward == m[1].a.forward) return false;
		if (!disjoin_segments(m[1], m[2])) return false;
	} else if (n == 2) {
		if (m[0].a.supplementary || m[1].a.supplementary) return false;
	} else return false;
	for (int s = 0; s < 2; ++s) if ((m[s].front() & 15) == C_H || (m[s].back() & 15) == C_H) return false; // anchors need their full sequence
	return true;
}

// the alignments of fragment g, normalised; false: the fragment is malformed and dropped. Sequence offsets in m[].a are global bytes into the pool.
ARB_HD bool normalised(const pool_view& p, u32 g, norm_slot* m, u32& n) {
	const arb_pool_fragment& f = p.frags[g];
	n = 0;
	if (f.count < 2 || f.count > 3) return false; // every rule below wants two or three alignments
	const u32 w = p.worker_of(g);
	for (i32 x = f.head; x >= 0 && n < 3; ++n) {
		norm_slot& s = m[n];
		s.a = p.alns[p.aln_base[w] + (u64) x];
		s.cig = p.cigars + p.cigar_base[w] + s.a.cigar_off; s.cnt = s.a.cigar_cnt; s.n_edits = 0;
		s.a.seq_off += p.seq_base[w];
		x = s.a.next;
	}
	return normalise_fragment(m, n, f.single_end != 0);
}
ARB_HD u32 seq_units(u32 seq_len) { return ((seq_len + 1) / 2 + 15) / 16; }

// sums of a launch: one atomic per warp
ARB_HD void add_total(unsigned long long* p, u32 v) {
#ifdef __CUDA_ARCH__
	const unsigned active = __activemask();
	const u32 s = __reduce_add_sync(active, v);
	if ((threadIdx.x & 31u) == (u32) (__ffs((int) active) - 1)) atomicAdd(p, (unsigned long long) s);
#else
	*p += v;
#endif
}

// 1. per fragment: does it survive normalisation, how many CIGAR operations, 16-byte sequence units and name bytes it brings, its first 16 name bytes
struct ft_normalise_fn {
	pool_view p; u32* keep; u32* n_cigar; u32* n_units; u32* n_name; u64* key0; u64* key1; unsigned long long* totals /* cigar ops, sequence units, name bytes */;
	ARB_HD void operator()(u32 g) const {
		norm_slot m[3]; u32 n = 0;
		const bool ok = normalised(p, g, m, n);
		u32 c = 0, u = 0, l = 0;
		if (ok) {
			for (u32 s = 0; s < n; ++s) { c += m[s].cnt; if (s < 2) u += seq_units(m[s].a.seq_len); }
			l = p.frags[g].name_len;
			key0[g] = p.name_word(g, 0); key1[g] = p.name_word(g, 1);
		}
		keep[g] = ok ? 1 : 0; n_cigar[g] = c; n_units[g] = u; n_name[g] = l;
		add_total(totals, c); add_total(totals + 1, u); add_total(totals + 2, l);
	}
};
struct ft_compact_fn { const u32* keep; const u32* at; u32* ids; ARB_HD void operator()(u32 g) const { if (keep[g]) ids[at[g]] = g; } };

// 2. name order: LSD passes of 32 bits; `part` selects the word and half the pass sorts by
struct ft_key_fn {
	const u64* key0; const u64* key1; const u32* order; u32* keys; u32 part; // 0 low half of key1, 1 high half of key1, 2 low half of key0, 3 high half of key0
	ARB_HD void operator()(u32 i) const { const u64 k = part < 2 ? key1[order[i]] : key0[order[i]]; keys[i] = (part & 1) ? (u32) (k >> 32) : (u32) k; }
};
struct ft_first_heads_fn { // positions where the first 16 bytes change
	const u64* key0; const u64* key1; const u32* order; u32* head; u32 n;
	ARB_HD void operator()(u32 i) const { head[i] = i == 0 || key0[order[i]] != key0[order[i - 1]] || key1[order[i]] != key1[order[i - 1]] ? 1 : 0; }
};
// Runs of equal keys are sorted again by the next name word. A round works on the positions that are still in runs of two or more (`pos`, ascending) and the
// run each one belongs to (`run`, ascending along `pos`).
struct ft_iota_fn { u32* v; ARB_HD void operator()(u32 i) const { v[i] = i; } };
struct ft_still_tied_fn { const u32* head; u32* tied; u32 m; ARB_HD void operator()(u32 k) const { tied[k] = !head[k] || (k + 1 < m && !head[k + 1]) ? 1 : 0; } };
struct ft_run_of_fn { const u32* head_scan; u32* run; ARB_HD void operator()(u32 k) const { run[k] = head_scan[k + 1]; } }; // inclusive count of run heads
struct ft_compact_tied_fn {
	const u32* tied; const u32* at; const u32* pos; const u32* run; u32* pos_out; u32* run_out;
	ARB_HD void operator()(u32 k) const { if (tied[k]) { pos_out[at[k]] = pos[k]; run_out[at[k]] = run[k]; } }
};
struct ft_tie_key_fn { // key of pass `part` for tied element perm[j]: low / high half of its name word, then its run
	pool_view p; const u32* order; const u32* pos; const u32* run; const u32* perm; u32* keys; u32 word, part;
	ARB_HD void operator()(u32 j) const {
		const u32 k = perm[j];
		if (part == 2) { keys[j] = run[k]; return; }
		const u64 v = p.name_word(order[pos[k]], word);
		keys[j] = part ? (u32) (v >> 32) : (u32) v;
	}
};
struct ft_tie_gather_fn { const u32* order; const u32* pos; const u32* perm; u32* ids; ARB_HD void operator()(u32 j) const { ids[j] = order[pos[perm[j]]]; } };
struct ft_tie_scatter_fn { // a run occupies the same positions before and after: the sorted elements go back to the positions in `pos`
	pool_view p; u32* order; const u32* pos; const u32* run; const u32* perm; const u32* ids; u32* head; u32 word;
	ARB_HD void operator()(u32 j) const {
		order[pos[j]] = ids[j];
		head[j] = j == 0 || run[perm[j]] != run[perm[j - 1]] || p.name_word(ids[j], word) != p.name_word(ids[j - 1], word) ? 1 : 0;
	}
};

// 3. sizes in name order (scanned into offsets by the driver)
struct ft_sizes_fn {
	const u32* order; const u32* n_cigar; const u32* n_units; const u32* n_name; u32* c; u32* u; u32* l;
	ARB_HD void operator()(u32 i) const { const u32 g = order[i]; c[i] = n_cigar[g]; u[i] = n_units[g]; l[i] = n_name[g]; }
};

// 4. the columns of fragment i (arb_soa_chunk layout), normalised again from the pools
struct ft_fill_fn {
	pool_view p; const u32* order; const u32* cig_at; const u32* unit_at; const u32* name_at; frag_view f; char* names; u64* name_off;
	ARB_HD void operator()(u32 i) const {
		const u32 g = order[i], n_frag = f.n;
		norm_slot m[3]; u32 n = 0;
		normalised(p, g, m, n); // true: only survivors are in `order`
		const arb_pool_fragment& fb = p.frags[g];
		f.n_aln[i] = (u8) n; f.fflags[i] = (fb.single_end ? FF_SINGLE_END : 0) | (fb.duplicate ? FF_DUPLICATE : 0); f.filter[i] = 0;
		u32 c = cig_at[i], sq = unit_at[i];
		for (u32 s = 0; s < 3; ++s) {
			const u32 x = s * n_frag + i;
			if (s >= n) { f.contig[x] = 0; f.start[x] = 0; f.end[x] = 0; f.aflags[x] = 0; f.cigar_off[x] = 0; f.cigar_cnt[x] = 0; if (s < 2) { f.seq_off[x] = 0; f.seq_len[x] = 0; } continue; }
			const norm_slot& a = m[s];
			f.contig[x] = a.a.contig; f.start[x] = a.a.start; f.end[x] = a.a.end;
			f.aflags[x] = (a.a.supplementary ? AF_SUPPLEMENTARY : 0) | (a.a.first_in_pair ? AF_FIRST_IN_PAIR : 0) | (a.a.forward ? AF_FORWARD : 0) | AF_PRED_AMBIGUOUS;
			f.cigar_off[x] = c; f.cigar_cnt[x] = (u16) a.cnt;
			for (u32 k = 0; k < a.cnt; ++k) f.cigar[c + k] = a.op(k);
			c += a.cnt;
			if (s < 2) {
				f.seq_off[x] = sq; f.seq_len[x] = (u16) a.a.seq_len;
				// whole 16-byte units: the bases, then zero bytes (the pool's sequences start 16-byte aligned)
				const u32 bytes = (a.a.seq_len + 1) / 2, units = seq_units(a.a.seq_len);
				const u8* src = p.seqs + a.a.seq_off; u8* dst = f.seq + (u64) sq * 16;
				for (u32 q = 0; q < units; ++q) {
					u32 w[4];
					const u32* s4 = (const u32*) (src + 16 * q);
					for (u32 k = 0; k < 4; ++k) {
						const u32 lo = 16 * q + 4 * k;
						w[k] = lo + 4 <= bytes ? s4[k] : lo >= bytes ? 0u : s4[k] & (0xFFFFFFFFu >> (8 * (lo + 4 - bytes)));
					}
					u32* d4 = (u32*) (dst + 16 * q);
					d4[0] = w[0]; d4[1] = w[1]; d4[2] = w[2]; d4[3] = w[3];
				}
				sq += units;
			}
		}
		u32 len; const char* s = p.name(g, len);
		char* d = names + name_at[i];
		for (u32 k = 0; k < len; ++k) d[k] = s[k];
		name_off[i] = name_at[i];
		if (i + 1 == n_frag) name_off[n_frag] = name_at[n_frag];
	}
};

// 5. multimappers: neighbours in name order that share the name up to the last comma
struct ft_same_name_fn {
	const char* names; const u64* name_off; u8* same;
	ARB_HD u64 stem_len(u32 i) const { const char* s = names + name_off[i]; const u64 l = name_off[i + 1] - name_off[i]; u64 k = l; while (k > 0 && s[k - 1] != ',') --k; return k > 0 ? k - 1 : l; }
	ARB_HD void operator()(u32 i) const {
		const u64 la = stem_len(i), lb = stem_len(i + 1);
		bool eq = la == lb;
		for (u64 k = 0; eq && k < la; ++k) eq = names[name_off[i] + k] == names[name_off[i + 1] + k];
		same[i] = eq ? 1 : 0;
	}
};
struct ft_multimapper_fn {
	const u8* same; u8* fflags;
	ARB_HD void operator()(u32 i) const {
		const bool before = i > 0 && same[i - 1];
		if (same[i] || before) fflags[i] |= FF_MULTIMAPPER;
		if (before) fflags[i] |= FF_SAME_NAME_AS_PREVIOUS;
	}
};

} // namespace arb
