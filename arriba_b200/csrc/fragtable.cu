// fragtable.cu -- the fragment table in name order, built on the device from the pools of the ingest workers (rules in fragtable_hd.h).
//
// The record loop of the ingest (host/ingest.cpp) leaves every worker with append-only pools. Here they are copied to the device and
//   1. every fragment is normalised into its slots or rejected; survivors report their CIGAR, sequence and name sizes and their first 16 name bytes;
//   2. the survivors are radix-sorted by those 16 bytes (four stable 32-bit passes); runs of equal keys are sorted again by the next 8 bytes of their
//      names, round after round, until no two neighbours are tied (names are unique);
//   3. exclusive scans in name order give the pool offsets;
//   4. one thread per fragment normalises it again and writes its columns, CIGARs, sequences and name;
//   5. neighbours with the same read name are flagged as multimappers.
// The table stays resident as if arb_push_chunk_begin had sent it; arb_get_fragment_table copies it back for the host-side consumers.
#include "engine.h"
#include "fragtable_hd.h"

namespace arb {

template <class T> static void copy_async(const exec_ctx& ex, T* dst, const T* src, size_t n, bool to_device) {
	if (!n) return;
#ifdef ARB_DEVICE_BUILD
	ARB_CUDA_CHECK(cudaMemcpyAsync(dst, src, n * sizeof(T), to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost, ex.stream));
#else
	(void) ex; (void) to_device;
	memcpy(dst, src, n * sizeof(T));
#endif
}

void engine::build_fragment_table(const arb_ingest_pool* pools, u32 n_pools, arb_fragment_table_sizes& sizes) {
	if (n_pools == 0 || !pools) throw arb_error("arb_build_fragment_table: no pools");
	ex.sync(); copy_ex.sync(); // kernels or copies of the previous sample may still use the buffers that are about to be overwritten
	stage_timer t_all(ex);
	// ---- the pools, worker after worker (sequences 16-byte aligned)
	std::vector<u64> name_base(n_pools), cigar_base(n_pools), seq_base(n_pools), aln_base(n_pools); std::vector<u32> frag_base((size_t) n_pools + 1);
	u64 names = 0, cigars = 0, seqs = 0, alns = 0, frags_total = 0;
	for (u32 w = 0; w < n_pools; ++w) {
		name_base[w] = names; cigar_base[w] = cigars; seq_base[w] = seqs; aln_base[w] = alns; frag_base[w] = (u32) frags_total;
		names += pools[w].n_name_bytes; cigars += pools[w].n_cigars; seqs += (pools[w].n_seq_bytes + 15) & ~(u64) 15; alns += pools[w].n_alns; frags_total += pools[w].n_frags;
	}
	if (frags_total >= 0xFFFFFFFFull) throw arb_error("chunk too large: more than 2^32 fragments");
	const u32 N = (u32) frags_total;
	frag_base[n_pools] = N;
	ft_names.ensure(names + 8); ft_cigars.ensure(cigars + 1); ft_seqs.ensure(seqs + 16); ft_alns.ensure(alns + 1); ft_frags.ensure((size_t) N + 1);
	ft_bases.ensure(4 * (size_t) n_pools); ft_frag_base.ensure((size_t) n_pools + 1);
	stage_timer t_h2d(ex);
	for (u32 w = 0; w < n_pools; ++w) {
		const arb_ingest_pool& q = pools[w];
		copy_async(ex, ft_names.ptr() + name_base[w], q.names, q.n_name_bytes, true);
		copy_async(ex, ft_cigars.ptr() + cigar_base[w], q.cigars, q.n_cigars, true);
		copy_async(ex, ft_seqs.ptr() + seq_base[w], q.seqs, q.n_seq_bytes, true);
		copy_async(ex, ft_alns.ptr() + aln_base[w], q.alns, q.n_alns, true);
		copy_async(ex, ft_frags.ptr() + frag_base[w], q.frags, q.n_frags, true);
	}
	std::vector<u64> bases(4 * (size_t) n_pools);
	for (u32 w = 0; w < n_pools; ++w) { bases[w] = name_base[w]; bases[n_pools + w] = cigar_base[w]; bases[2 * n_pools + w] = seq_base[w]; bases[3 * n_pools + w] = aln_base[w]; }
	copy_async(ex, ft_bases.ptr(), bases.data(), bases.size(), true);
	copy_async(ex, ft_frag_base.ptr(), frag_base.data(), frag_base.size(), true);
	timings.h2d_ms = sizes.upload_ms = t_h2d.stop(); // the pool upload: the columns of the table never cross PCIe towards the device
	timings.h2d_bytes = names + cigars * 4 + seqs + alns * sizeof(arb_pool_alignment) + (u64) N * sizeof(arb_pool_fragment) + bases.size() * 8 + frag_base.size() * 4;
	pool_view p;
	p.names = ft_names.ptr(); p.cigars = ft_cigars.ptr(); p.seqs = ft_seqs.ptr(); p.alns = ft_alns.ptr(); p.frags = ft_frags.ptr();
	p.name_base = ft_bases.ptr(); p.cigar_base = ft_bases.ptr() + n_pools; p.seq_base = ft_bases.ptr() + 2 * (size_t) n_pools; p.aln_base = ft_bases.ptr() + 3 * (size_t) n_pools;
	p.frag_base = ft_frag_base.ptr(); p.n_workers = n_pools;

	// ---- 1. normalisation
	dbuf<u32> keep((size_t) N + 1), at((size_t) N + 1), n_cigar(N), n_units(N), n_name(N); dbuf<u64> key0(N), key1(N); dbuf<u64> totals(4);
	totals.zero(ex, 4);
	ft_normalise_fn nf = {p, keep.ptr(), n_cigar.ptr(), n_units.ptr(), n_name.ptr(), key0.ptr(), key1.ptr(), (unsigned long long*) totals.ptr()};
	for_each(ex, N, nf);
	exclusive_scan_u32(ex, keep.ptr(), at.ptr(), N);
	u64 tot[4] = {0, 0, 0, 0}; totals.download(ex, tot, 3);
	u32 n = 0; at.download(ex, &n, 1, N);
	sizes.n_rejected = N - n;
	if (tot[0] > 0xFFFFFFFFull || tot[1] > 0xFFFFFFFFull) throw arb_error("chunk too large: more than 2^32 CIGAR operations or 64 GiB of sequence");
	if (tot[2] > 0xFFFFFFFFull) throw arb_error("chunk too large: more than 4 GiB of read names");
	dbuf<u32> order((size_t) n + 1), keys((size_t) n + 1), tk((size_t) n + 1), tv((size_t) n + 1);
	ft_compact_fn cf = {keep.ptr(), at.ptr(), order.ptr()};
	for_each(ex, N, cf);

	// ---- 2. name order
	for (u32 part = 0; part < 4; ++part) {
		ft_key_fn kf = {key0.ptr(), key1.ptr(), order.ptr(), keys.ptr(), part};
		for_each(ex, n, kf);
		radix_sort_pairs_u32(ex, keys.ptr(), order.ptr(), tk.ptr(), tv.ptr(), n, 32);
	}
	u32 rounds = 0;
	{
		dbuf<u32> head((size_t) n + 1), scan((size_t) n + 1), pos((size_t) n + 1), run((size_t) n + 1), pos2((size_t) n + 1), run2((size_t) n + 1), tied((size_t) n + 1), perm((size_t) n + 1), ids((size_t) n + 1);
		ft_first_heads_fn hf = {key0.ptr(), key1.ptr(), order.ptr(), head.ptr(), n};
		for_each(ex, n, hf);
		// round 0 works on every position
		ft_iota_fn io = {pos.ptr()}; for_each(ex, n, io);
		exclusive_scan_u32(ex, head.ptr(), scan.ptr(), n);
		ft_run_of_fn rf = {scan.ptr(), run.ptr()}; for_each(ex, n, rf);
		u32 m = n;
		for (u32 word = 2; m > 1; ++word) {
			ft_still_tied_fn tf = {head.ptr(), tied.ptr(), m}; for_each(ex, m, tf);
			exclusive_scan_u32(ex, tied.ptr(), scan.ptr(), m);
			u32 m2 = 0; scan.download(ex, &m2, 1, m);
			if (m2 == 0) break;
			if (word > 2 + 1024 / 8) throw arb_error("fragment names are not unique"); // BAM names have at most 254 bytes
			ft_compact_tied_fn ctf = {tied.ptr(), scan.ptr(), pos.ptr(), run.ptr(), pos2.ptr(), run2.ptr()}; for_each(ex, m, ctf);
			pos.swap(pos2); run.swap(run2); m = m2;
			++rounds;
			ft_iota_fn ip = {perm.ptr()}; for_each(ex, m, ip);
			for (u32 part = 0; part < 3; ++part) {
				ft_tie_key_fn kf = {p, order.ptr(), pos.ptr(), run.ptr(), perm.ptr(), keys.ptr(), word, part};
				for_each(ex, m, kf);
				radix_sort_pairs_u32(ex, keys.ptr(), perm.ptr(), tk.ptr(), tv.ptr(), m, 32);
			}
			ft_tie_gather_fn gf = {order.ptr(), pos.ptr(), perm.ptr(), ids.ptr()}; for_each(ex, m, gf);
			ft_tie_scatter_fn sf = {p, order.ptr(), pos.ptr(), run.ptr(), perm.ptr(), ids.ptr(), head.ptr(), word}; for_each(ex, m, sf);
			exclusive_scan_u32(ex, head.ptr(), scan.ptr(), m);
			ft_run_of_fn rf2 = {scan.ptr(), run.ptr()}; for_each(ex, m, rf2);
		}
	}
	sizes.tie_rounds = rounds; tie_rounds = rounds;

	// ---- 3. offsets in name order
	dbuf<u32> cig_at((size_t) n + 1), unit_at((size_t) n + 1), name_at((size_t) n + 1);
	ft_sizes_fn zf = {order.ptr(), n_cigar.ptr(), n_units.ptr(), n_name.ptr(), cig_at.ptr(), unit_at.ptr(), name_at.ptr()};
	for_each(ex, n, zf);
	exclusive_scan_u32(ex, cig_at.ptr(), cig_at.ptr(), n); exclusive_scan_u32(ex, unit_at.ptr(), unit_at.ptr(), n); exclusive_scan_u32(ex, name_at.ptr(), name_at.ptr(), n);

	// ---- 4. the columns, straight into the resident table
	const u64 n_cigar_ops = tot[0] + 1, n_seq_bytes = tot[1] * 16 + 16, n_name_bytes = tot[2]; // one zero operation and one zero unit behind the pools
	frags.n = n;
	frags.n_aln.ensure(n); frags.fflags.ensure(n); frags.filter.ensure(n);
	frags.contig.ensure(3 * (size_t) n); frags.start.ensure(3 * (size_t) n); frags.end.ensure(3 * (size_t) n); frags.aflags.ensure(3 * (size_t) n);
	frags.cigar_off.ensure(3 * (size_t) n); frags.cigar_cnt.ensure(3 * (size_t) n); frags.seq_off.ensure(2 * (size_t) n); frags.seq_len.ensure(2 * (size_t) n);
	frags.cigar.ensure(n_cigar_ops); frags.seq.ensure(n_seq_bytes);
	ft_out_names.ensure(n_name_bytes + 1); ft_out_name_off.ensure((size_t) n + 1);
	frag_view fv = frags.view();
	ft_fill_fn ff = {p, order.ptr(), cig_at.ptr(), unit_at.ptr(), name_at.ptr(), fv, ft_out_names.ptr(), ft_out_name_off.ptr()};
	for_each(ex, n, ff);
#ifdef ARB_DEVICE_BUILD
	ARB_CUDA_CHECK(cudaMemsetAsync(frags.cigar.ptr() + tot[0], 0, 4, ex.stream));
	ARB_CUDA_CHECK(cudaMemsetAsync(frags.seq.ptr() + tot[1] * 16, 0, 16, ex.stream));
#else
	frags.cigar.ptr()[tot[0]] = 0; memset(frags.seq.ptr() + tot[1] * 16, 0, 16);
#endif
	if (n == 0) { const u64 zero = 0; copy_async(ex, ft_out_name_off.ptr(), &zero, 1, true); }

	// ---- 5. multimappers
	if (n > 1) {
		dbuf<u8> same(n); same.zero(ex, n);
		ft_same_name_fn sn = {ft_out_names.ptr(), ft_out_name_off.ptr(), same.ptr()};
		for_each(ex, n - 1, sn);
		ft_multimapper_fn mf = {same.ptr(), frags.fflags.ptr()};
		for_each(ex, n, mf);
	}
	table_resident(ex, n_cigar_ops, n_seq_bytes);
	sizes.build_ms = t_all.stop();
	sizes.n_fragments = n; sizes.n_cigar = n_cigar_ops; sizes.n_seq_bytes = n_seq_bytes; sizes.n_name_bytes = n_name_bytes;
	ft_n_name_bytes = n_name_bytes;
}

void engine::get_fragment_table(const arb_fragment_columns& o) {
	const u32 n = frags.n;
	// the columns the host reads first go first; the sequence pool last
	copy_async(ex, o.n_aln, frags.n_aln.ptr(), n, false); copy_async(ex, o.fflags, frags.fflags.ptr(), n, false); copy_async(ex, o.filter, frags.filter.ptr(), n, false);
	copy_async(ex, o.contig, frags.contig.ptr(), 3 * (size_t) n, false); copy_async(ex, o.start, frags.start.ptr(), 3 * (size_t) n, false); copy_async(ex, o.end, frags.end.ptr(), 3 * (size_t) n, false);
	copy_async(ex, o.aflags, frags.aflags.ptr(), 3 * (size_t) n, false);
	copy_async(ex, o.name_off, ft_out_name_off.ptr(), (size_t) n + 1, false); copy_async(ex, o.names, ft_out_names.ptr(), ft_n_name_bytes, false);
	copy_async(ex, o.cigar_off, frags.cigar_off.ptr(), 3 * (size_t) n, false); copy_async(ex, o.cigar_cnt, frags.cigar_cnt.ptr(), 3 * (size_t) n, false);
	copy_async(ex, o.seq_off, frags.seq_off.ptr(), 2 * (size_t) n, false); copy_async(ex, o.seq_len, frags.seq_len.ptr(), 2 * (size_t) n, false);
	copy_async(ex, o.cigar, frags.cigar.ptr(), push_cigar_ops, false);
	copy_async(ex, o.seq, frags.seq.ptr(), frags.n_seq_bytes, false);
	ex.sync();
}

} // namespace arb
