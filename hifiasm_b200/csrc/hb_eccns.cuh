// hb_eccns.cuh — window consensus of an error-correction round (SURVEY.md §8 row a14): wcns_gen (ecovlp.cpp:2293) per read.
//
// What the reference does with the same-haplotype overlaps (is_match == 1) of a read after phasing and dedup_chains:
//   * every aligned window of every such overlap becomes an entry (overlap, window, cigar cursor), sorted by query start (2297-2385);
//   * the read is swept in 512-column blocks; per block the entries that cover it vote per column: wcns_vote (2185) counts
//     (match, total) per base column and per gap in front of a column (extract_sub_cigar_mm 283) and keeps the columns where the
//     read's own base wins (> 0.500001 of the votes and more than the rest, at least 3 voters) — or where fewer than 3 voters exist;
//   * maximal runs of kept columns are anchors (push_cns_anchor 2109): they go to the edit script as match runs, and the stretch
//     between two anchors is corrected by a vote over the sub-alignments that span it (cns_gen0 1159 -> extract_sub_cigar_ii 365:
//     stretches of <= 6 columns whose most frequent (cigar, bases) variant has the majority), else by a small graph consensus
//     (cns_gen_full 1919).  THE GRAPH CONSENSUS IS NOT BUILT YET: a read that needs it is reported (need_full) and gets no script.
// The edit script is the reference's encoding (push_trace_bp_f, Levenshtein_distance.h:640; see hb_ecround.cuh).
// One thread per read; all state lives in per-read slices of HBM scratch.  The reference's quirks are kept on purpose and marked.
#pragma once
#include "hb_common.cuh"
#include "hb_ecaln.cuh"
#include "hb_ecround.cuh"

#define HB_CNS_WL 512        // block length of the sweep (wcns_gen's wl, ecovlp.cpp:3309)
#define HB_CNS_VOTE_LEN 6    // simp_vote_len, ecovlp.cpp:362

struct CnsEnt { uint32_t ov, wid, xoff, yoff; int32_t coff; };  // ul_ov_t as wcns_gen uses it (ovlp_id, cur_wid, cur_xoff, cur_yoff, cur_coff; bd = 0, ylen = 0)
struct CnsOv { const hb_wl_t *w; uint32_t wn, y_id, rev; };    // a same-haplotype overlap: its step-C window list (cigars in the shared pool)
struct CnsIt { const uint32_t *srt; uint32_t *act; int64_t i, srt_n, act_n, rr, ru; uint64_t mms, mme; }; // cc_idx_t (274-279): act = idx->a + srt_n
struct CnsG;
struct CnsCtx {
	DevReads R; RdView q; int64_t ql; CnsG *g;   // g: arena of the graph consensus (hb_eccns_full.cuh); NULL = voted path only
	const CnsOv *ov; const uint16_t *pool; CnsEnt *ent;
	CnsIt A, B; uint64_t *ct; uint32_t *b32; uint32_t b32_n;
	uint16_t *out; uint32_t out_n, out_cap; int32_t ax_start, ax_end; int has_win;   // aux_o's single window: the script under construction
	int ovf, need_full;
};

// push_trace_bp_f, Levenshtein_distance.h:640-670
HB_HD void hb_sc_push(CnsCtx &C, uint32_t c, uint32_t bq, uint32_t bt, uint32_t len, uint32_t is_append)
{
	c &= 0xffff; bq &= 0xffff; bt &= 0xffff;
	uint32_t c0, bq0, bt0, len0, mm;
	if (c == 3) { bt = bq; bq = HB_SC_NONE; }
	if (is_append && C.out_n) {
		bq0 = bq; bt0 = bt; const uint16_t in = C.out[C.out_n - 1];
		c0 = in >> 14;
		if (c0 == 2 || c0 == 3) { bt0 = (in >> 12) & 3; len0 = in & 0xfff; }
		else if (c0 == 1) { bt0 = (in >> 12) & 3; bq0 = (in >> 10) & 3; len0 = in & 0x3ff; }
		else len0 = in & 0x3fff;
		if (c == c0 && bq == bq0 && bt == bt0) { C.out_n--; len += len0; }
	}
	uint32_t w = c << 14;
	if (c == 2 || c == 3) { mm = 0xfff; w += (bt & 3) << 12; }
	else if (c == 1) { mm = 0x3ff; w += (bt & 3) << 12; w += (bq & 3) << 10; }
	else mm = 0x3fff;
	while (len >= mm) { if (C.out_n < C.out_cap) C.out[C.out_n] = (uint16_t)(w + mm); else C.ovf = 1; C.out_n++; len -= mm; }
	if (len) { if (C.out_n < C.out_cap) C.out[C.out_n] = (uint16_t)(w + len); else C.ovf = 1; C.out_n++; }
	if (C.ovf && C.out_n > C.out_cap) C.out_n = C.out_cap; // keep the cursor inside the buffer; the read is redone with a larger one
}

// iter_cc_idx_t, ecovlp.cpp:1055-1100: the entries that overlap [s, e), kept as a list that is pruned (is_reduce) and extended in query order
HB_HD uint32_t hb_cns_iter(CnsCtx &C, CnsIt &z, int64_t s, int64_t e, int64_t is_reduce, int is_insert)
{
	if (z.ru == 0) {
		int64_t q0, q1, os, oe;
		if (is_reduce) {
			int64_t rm_n = 0;
			for (int64_t m = 0; m < z.act_n; m++) {
				const CnsEnt &cp = C.ent[z.act[m]]; const hb_wl_t &w = C.ov[cp.ov].w[cp.wid];
				q0 = w.x_start; q1 = (int64_t)w.x_end + 1; os = q0 > s ? q0 : s; oe = q1 < e ? q1 : e;
				if (oe > os || (is_insert && s == e && s >= q0 && s <= q1)) z.act[rm_n++] = z.act[m];
			}
			z.act_n = rm_n;
		}
		for (; z.i < z.srt_n; ++z.i) {
			const CnsEnt &cp = C.ent[z.srt[z.i]]; const hb_wl_t &w = C.ov[cp.ov].w[cp.wid];
			q0 = w.x_start; q1 = (int64_t)w.x_end + 1;
			if (q0 > e) break;
			if (!is_insert && q0 >= e) break;
			os = q0 > s ? q0 : s; oe = q1 < e ? q1 : e;
			if (oe > os || (is_insert && s == e && s >= q0 && s <= q1)) z.act[z.act_n++] = z.srt[z.i];
		}
	} else z.ru = 0;
	return (uint32_t)z.act_n;
}


// extract_sub_cigar_ii, ecovlp.cpp:365-517: the variant one window alignment proposes for the stretch [iws, iwe) (s..e = its part inside the
// window): [cigar length:4][cigar:12][base count:4][bases:12], or -1 when the alignment does not span the stretch or the variant is longer than 6
HB_HD uint32_t hb_cns_sub_ii(CnsCtx &C, CnsEnt &p, int64_t s, int64_t e, int64_t iws, int64_t iwe)
{
	const CnsOv &z = C.ov[p.ov]; const hb_wl_t &w = z.w[p.wid];
	int64_t xk = p.xoff, yk = p.yoff, ck = p.coff, os, oe, ol, ii0, ii1, it0, it1; uint32_t res;
	const int64_t s0 = w.x_start, e0 = (int64_t)w.x_end + 1;
	if (s < s0) s = s0; if (e > e0) e = e0;
	if (s > e) return 0xffffffffu;
	os = s > s0 ? s : s0; oe = e < e0 ? e : e0;
	if (oe < os) return 0xffffffffu;
	if (!((s0 < iws || s0 == 0) && (e0 > iwe || e0 == C.ql))) return 0xffffffffu;
	const uint16_t *cg = C.pool + w.cidx; const int64_t cn = w.clen;
	if (!cn) return 0xffffffffu;
	uint32_t op; int64_t ws, we, wts, wte, ovlp, cc = 0, cci;
	if (ck < 0 || ck > cn) { ck = 0; xk = w.x_start; yk = w.y_start; }
	while (ck > 0 && xk >= s) { --ck; op = cg[ck] >> 14; if (op != 2) xk -= cg[ck] & 0x3fff; if (op != 3) yk -= cg[ck] & 0x3fff; }
	ii0 = ii1 = it0 = it1 = -1; res = 0; cc = 0;
	while (ck < cn && xk < e) {
		ws = xk; wts = yk; op = cg[ck] >> 14; ol = cg[ck] & 0x3fff;
		if (op != 2) xk += ol; if (op != 3) yk += ol;
		ck++; we = xk; wte = yk;
		os = s > ws ? s : ws; oe = e < we ? e : we; ovlp = oe > os ? oe - os : 0;
		if (s == e) { if (op != 0 || ws >= s || we <= e || e != iwe || s != iws) continue; }
		else { if (op != 2) { if (!ovlp) continue; } else { if (ws < s || ws >= e) continue; } }
		if (ii0 == -1) { ii0 = os; it0 = op < 2 ? os - ws + wts : wts; }
		ii1 = oe; it1 = op < 2 ? oe - ws + wts : wte;
		if (op != 2) ol = oe - os;
		cc += ol;
		if (cc <= HB_CNS_VOTE_LEN) for (cci = 0; cci < ol; cci++) { res <<= 2; res |= op; }
	}
	while (ck < cn && xk <= e) {
		ws = xk; wts = yk; op = cg[ck] >> 14; ol = cg[ck] & 0x3fff;
		if (op != 2) break;
		yk += ol; ck++; we = xk; wte = yk;
		if (ws >= s && ws <= e) {
			if (ii0 == -1) { ii0 = ws; it0 = wts; }
			ii1 = we; it1 = wte;
			cc += ol;
			if (cc <= HB_CNS_VOTE_LEN) for (cci = 0; cci < ol; cci++) { res <<= 2; res |= op; }
		}
	}
	if (cc <= HB_CNS_VOTE_LEN && ii1 >= ii0 && ii1 - ii0 <= HB_CNS_VOTE_LEN && it1 >= it0 && it1 - it0 <= HB_CNS_VOTE_LEN) {
		if (ii0 == iws && ii1 == iwe) {
			uint32_t o16 = (uint32_t)cc & 0xffff; o16 = (o16 << 12) & 0xffff; res |= o16; // `op` is a uint16_t in the reference
			res <<= 16; cc = it1 - it0; o16 = 0;
			if (cc > 0) {
				const RdView T = hb_rd_view(C.R, z.y_id, z.rev);
				for (cci = 0; cci < cc; cci++) { o16 = (o16 << 2) & 0xffff; const int b = T.at(it0 + cci); o16 |= (uint32_t)(b == 4 ? 5 : b); } // seq_nt6_table gives an N the code 5 (Process_Read.cpp:12): it spills into the next base's bits, as in the reference
			}
			res |= o16;
			o16 = (uint32_t)(it1 - it0) & 0xffff; o16 = (o16 << 12) & 0xffff; res |= o16;
		} else res = 0xffffffffu;
	} else res = 0xffffffffu;
	p.xoff = (uint32_t)xk; p.yoff = (uint32_t)yk; p.coff = (int32_t)ck;
	return res;
}

HB_HD bool hb_cns_pass(uint64_t oc0, uint64_t oc1, uint64_t occ_tot, double occ_max)
{ return (double)oc0 > (double)oc1 * occ_max && oc0 > oc1 - oc0 && oc1 >= occ_tot && oc0 > 1; }

// small in-place sort of 32-bit values (radix_sort_ec32 on bare keys: any sort gives the same array)
HB_HD void hb_sort32(uint32_t *a, uint32_t n)
{ for (uint32_t i = 1; i < n; i++) { const uint32_t v = a[i]; uint32_t j = i; while (j > 0 && a[j - 1] > v) { a[j] = a[j - 1]; j--; } a[j] = v; } }

// cns_gen0, ecovlp.cpp:1159-1218: vote over the variants of the stretch [s, e) (s == e: an insertion site); 1 + *rc when one variant has the majority
HB_HD int hb_cns_gen0(CnsCtx &C, int64_t s, int64_t e, uint32_t *rc)
{
	if (e > s + HB_CNS_VOTE_LEN) return 0;
	CnsIt &idx = C.B; uint64_t an = 0, oc0, oc1; C.b32_n = 0;
	const uint32_t id_n = hb_cns_iter(C, idx, s, e, idx.rr, s == e ? 1 : 0);
	idx.rr = 0;
	for (uint32_t k = 0; k < id_n; k++) {
		CnsEnt &p = C.ent[idx.act[k]]; const hb_wl_t &w = C.ov[p.ov].w[p.wid];
		const int64_t q0 = w.x_start, q1 = (int64_t)w.x_end + 1;
		if (q1 <= e) idx.rr = 1;
		const int64_t os = q0 > s ? q0 : s, oe = q1 < e ? q1 : e;
		if (oe > os || (s == e && s > q0 && s < q1)) {
			const uint32_t m = hb_cns_sub_ii(C, p, os, oe, s, e); an++;
			if (m != 0xffffffffu) C.b32[C.b32_n++] = m;
		}
	}
	oc0 = C.b32_n; oc1 = an + 1;
	if (hb_cns_pass(oc0, oc1, 3, 0.500001)) {
		hb_sort32(C.b32, C.b32_n); an = 0; const uint32_t *a = 0;
		for (uint32_t k = 1, l = 0; k <= C.b32_n; ++k) if (k == C.b32_n || C.b32[k] != C.b32[l]) { if (k - l > an) { an = k - l; a = C.b32 + l; } l = k; }
		oc0 = an;
		if (hb_cns_pass(oc0, oc1, 3, 0.500001)) { *rc = a[0]; return 1; }
	}
	idx.ru = 1;
	return 0;
}

// push_correct0_fhc, ecovlp.cpp:1977-2016: a match run of len0, or the variant rc written op by op (qoff = start of the stretch on the read)
HB_HD uint64_t hb_cns_push0(CnsCtx &C, uint32_t len0, uint32_t rc, int64_t qoff)
{
	uint64_t nec = 0;
	if (len0 != 0xffffffffu) hb_sc_push(C, 0, HB_SC_NONE, HB_SC_NONE, len0, C.out_n > 0 ? 1 : 0);
	else if (rc != 0xffffffffu) {
		const uint32_t cc = (rc << 4) >> 20, cn = rc >> 28, bc = (rc << 20) >> 20, bn = (rc << 16) >> 28; uint32_t btk = 0, bqk = 0;
		for (uint32_t ck = 0; ck < cn; ck++) {
			const uint32_t cp = (cc >> ((cn - 1 - ck) << 1)) & 3; uint32_t bqp = 0xffffffffu, btp = 0xffffffffu;
			if (cp != 3) { btp = (bc >> ((bn - 1 - btk) << 1)) & 3; btk++; }
			if (cp != 2) { const int b = C.q.at(qoff + bqk); bqp = (uint32_t)(b == 4 ? 5 : b); bqk++; } // seq_nt6_table: N -> 5, stored as 5 & 3
			hb_sc_push(C, cp, bqp, btp, 1, C.out_n > 0 ? 1 : 0);
			if (cp != 0) nec++;
		}
	}
	return nec;
}

// cns_gen_full (hb_eccns_full.cuh); sets C.need_full = 2 when the arena is too small.  Out of line: inlined into k_ec_cns_w<true>, the one kernel
// that calls it, the graph code kept cicc (CUDA 12.9) busy for a quarter of an hour; as a call it compiles in seconds.
HB_HD_NI uint64_t hb_cns_full_(CnsCtx &C, int64_t s0, int64_t e0);
// push_cns_anchor, ecovlp.cpp:2109-2163
template <bool GRAPH> HB_HD uint64_t hb_cns_anchor(CnsCtx &C, uint64_t s, uint64_t e, int is_tail)
{
	if (!is_tail && s >= e) return 0;
	uint64_t e0 = 0, nec = 0; uint32_t rc;
	if (C.has_win) e0 = (uint64_t)((int64_t)C.ax_end + 1);
	if (s == e && is_tail == 1 && s == e0) return 0;
	if (!C.has_win) { C.has_win = 1; C.ax_start = -1; C.ax_end = -1; }
	if ((!is_tail && s > 0) || (is_tail && s > e0)) {
		if (hb_cns_gen0(C, (int64_t)e0, (int64_t)s, &rc)) {
			if (C.ax_start == -1 || C.ax_end == -1) { C.ax_start = (int32_t)e0; C.ax_end = (int32_t)s - 1; }
			nec += hb_cns_push0(C, 0xffffffffu, rc, (int64_t)e0);
		} else {
			if (!GRAPH || !C.g) { C.need_full = 1; return nec; } // no graph arena in this launch (GRAPH = false compiles the graph code out): the read is redone by the launch that has one
			nec += hb_cns_full_(C, (int64_t)e0, (int64_t)s);
			if (C.need_full) return nec;
		}
		C.ax_end = (int32_t)s - 1;
	}
	if (C.ax_start == -1 || C.ax_end == -1) { C.ax_start = (int32_t)s; C.ax_end = (int32_t)e - 1; }
	nec += hb_cns_push0(C, (uint32_t)(e - s), 0xffffffffu, 0);
	C.ax_end = (int32_t)e - 1;
	return nec;
}



// =====================================================================================================================================
// The same consensus with one WARP per read (hb_warp.cuh).  What changes is the shape of the work, not its result:
//   * the pile-up of a 512-column block — wcns_vote's first loop, which in the reference (and in the one-thread form kept in tests/hostemu/seq_ref.h) touches two counters per
//     column per covering alignment — becomes RANGE UPDATES on a difference array in shared memory: a lane owns a covering alignment, walks its
//     cigar RUNS and adds +v / -v at the two ends of the word range a run votes on (the reference's misplaced count-array offset, os - s WORDS,
//     only shifts where the range lands: a range of words base + 2 (t - s) + c is contiguous inside its parity class, so there is one
//     difference array per parity); one warp scan turns the differences into the per-column (match << 32 | voters) words;
//   * the per-column majority tests run one column per lane and leave two 512-bit masks (column kept / an insertion in front of it);
//   * lane 0 walks the masks run by run (count-trailing-zeros over 64-bit words), so the sequential part of a block is proportional to the
//     number of anchors, not of columns, and only there calls the reference's stretch vote (hb_cns_gen0) and script writer.
// =====================================================================================================================================
#include "hb_warp.cuh"
#define HB_CNS_DW 560                       // words of one parity class: 513 used, stored with one pad word per 16 (shared-memory banks)
#define HB_CNS_SMEM_WORDS (2 * HB_CNS_DW + 16) // per warp: two difference arrays + the two masks
HB_HD uint32_t hb_cns_dix(int64_t k) { return (uint32_t)(k + (k >> 4)); }

// extract_sub_cigar_mm (ecovlp.cpp:283-360) as range updates.  base = the word offset the reference adds to the count array (os - s of the block)
HB_HD void hb_cns_sub_mm_d(CnsCtx &C, CnsEnt &p, int64_t s, int64_t e, int64_t base, uint64_t *D)
{
	const hb_wl_t &w = C.ov[p.ov].w[p.wid];
	int64_t xk = p.xoff, yk = p.yoff, ck = p.coff, os, oe;
	const int64_t s0 = w.x_start, e0 = (int64_t)w.x_end + 1;
	if (s < s0) s = s0; if (e > e0) e = e0;
	if (s >= e) return;
	const uint16_t *cg = C.pool + w.cidx; const int64_t cn = w.clen;
	if (!cn) return;
	int64_t op, ws, we, ovlp;
	auto radd = [&](int64_t c, int64_t a, int64_t b, uint64_t v) { // words base + 2 (t - s) + c, t in [a, b)
		const int64_t w0 = base + c, h = w0 >> 1; uint64_t *d = D + (w0 & 1) * HB_CNS_DW;
		hb_atom_add64(d + hb_cns_dix(h + (a - s)), v); hb_atom_add64(d + hb_cns_dix(h + (b - s)), 0 - v);
	};
	if (ck < 0 || ck > cn) { ck = 0; xk = w.x_start; yk = w.y_start; }
	while (ck > 0 && xk >= s) { --ck; op = cg[ck] >> 14; if (op != 2) xk -= cg[ck] & 0x3fff; if (op != 3) yk -= cg[ck] & 0x3fff; }
	while (ck < cn && xk < e) {
		ws = xk; op = cg[ck] >> 14;
		if (op != 2) xk += cg[ck] & 0x3fff; if (op != 3) yk += cg[ck] & 0x3fff;
		ck++; we = xk;
		os = s > ws ? s : ws; oe = e < we ? e : we; ovlp = oe > os ? oe - os : 0;
		if (op != 2) { if (!ovlp) continue; } else { if (ws < s || ws >= e) continue; }
		if (op != 2) {
			const uint64_t v = op == 0 ? 0x100000001ULL : 1ULL;
			radd(0, os, oe, v);
			const int64_t a = os > ws ? os : os + 1; // the gap in front of the run's first column belongs to the previous run
			if (a < oe) radd(1, a, oe, v);
		} else radd(1, ws, ws + 1, 1);
	}
	p.xoff = (uint32_t)xk; p.yoff = (uint32_t)yk; p.coff = (int32_t)ck;
}

// number of consecutive bits equal to `want` from bit k on (bits >= n do not count)
HB_HD uint32_t hb_bits_run(const uint64_t *m, uint32_t k, uint32_t n, int want)
{
	const uint32_t k0 = k;
	while (k < n) {
		uint64_t v = m[k >> 6]; if (want) v = ~v; // bits that differ from `want`
		v >>= (k & 63);                           // (the zeros shifted in at the top read as "equal": a set bit is always inside the word)
		if (v) { k += (uint32_t)hb_ctz64(v); break; }
		k += 64 - (k & 63);
	}
	if (k > n) k = n;
	return k - k0;
}

// wcns_vote for a warp.  S = the warp's shared-memory words (HB_CNS_SMEM_WORDS).  Lane 0 owns the sequential state in C; every lane returns rr / sees need_full.
template <bool GRAPH> HB_HD int64_t hb_cns_vote_w(CnsCtx &C, uint64_t *S, uint32_t id_n, uint64_t s, uint64_t e, uint64_t *nec, int *need_full)
{
	const int lane = hb_lane(); uint64_t *D = S, *mP = S + 2 * HB_CNS_DW, *mI = mP + 8; const uint64_t wl = e - s;
	for (uint32_t k = lane; k < HB_CNS_SMEM_WORDS; k += HB_WS) S[k] = 0;
	hb_wsync();
	bool rrl = false;
	for (uint32_t k = lane; k < id_n; k += HB_WS) {
		CnsEnt &p = C.ent[C.A.act[k]]; const hb_wl_t &w = C.ov[p.ov].w[p.wid];
		const uint64_t q0 = (uint64_t)(int64_t)w.x_start, q1 = (uint64_t)((int64_t)w.x_end + 1);
		if (q1 <= e) rrl = true;
		const uint64_t os = q0 > s ? q0 : s, oe = q1 < e ? q1 : e;
		if (oe > os) hb_cns_sub_mm_d(C, p, (int64_t)os, (int64_t)oe, (int64_t)(os - s), D);
	}
	const int64_t rr = hb_any(rrl) ? 1 : 0;
	hb_wsync();
	{ // differences -> counts -> the two masks
		const uint32_t per = HB_CNS_WL / HB_WS, k0 = (uint32_t)lane * per; uint64_t a0 = 0, a1 = 0, t0, t1;
		for (uint32_t j = 0; j < per; j++) { a0 += D[hb_cns_dix(k0 + j)]; a1 += D[HB_CNS_DW + hb_cns_dix(k0 + j)]; }
		uint64_t c0 = hb_wscan64(a0, &t0), c1 = hb_wscan64(a1, &t1), accP = 0, accI = 0; int cw = -1;
		for (uint32_t j = 0; j < per; j++) {
			const uint32_t k = k0 + j; c0 += D[hb_cns_dix(k)]; c1 += D[HB_CNS_DW + hb_cns_dix(k)];
			if (k >= wl) break;
			if ((int)(k >> 6) != cw) { if (cw >= 0) { if (accP) hb_atom_or64(mP + cw, accP); if (accI) hb_atom_or64(mI + cw, accI); } cw = (int)(k >> 6); accP = accI = 0; }
			uint64_t oc0 = (c0 >> 32) + 1, oc1 = (uint32_t)c0 + 1;
			if (hb_cns_pass(oc0, oc1, 3, 0.500001) || oc1 < 3) {
				accP |= 1ULL << (k & 63);
				oc0 = (c1 >> 32) + 1; oc1 = (uint32_t)c1 + 1;
				if (!(hb_cns_pass(oc0, oc1, 3, 0.500001) || oc1 < 3)) accI |= 1ULL << (k & 63);
			}
		}
		if (cw >= 0) { if (accP) hb_atom_or64(mP + cw, accP); if (accI) hb_atom_or64(mI + cw, accI); }
	}
	hb_wsync();
	int nf = 0;
	if (lane == 0) {
		CnsIt &occ = C.B; uint64_t os = occ.mms, oe = occ.mme; uint32_t k = 0; uint64_t mC[8];
		for (int i = 0; i < 8; i++) mC[i] = mP[i] & ~mI[i];
#define HB_CNS_FLUSH() do { if (oe > os && os != (uint64_t)-1) { *nec += hb_cns_anchor<GRAPH>(C, os, oe, 0); if (C.need_full) { nf = 1; } } } while (0)
		while (k < wl && !nf) {
			if ((mP[k >> 6] >> (k & 63)) & 1) {
				if ((mI[k >> 6] >> (k & 63)) & 1) { HB_CNS_FLUSH(); if (nf) break; os = oe = (uint64_t)-1; }
				if (s + k == oe) { const uint32_t r = hb_bits_run(mC, k, (uint32_t)wl, 1); oe += r; k += r; } // columns kept with nothing inserted in front of them extend the anchor
				else { HB_CNS_FLUSH(); if (nf) break; os = s + k; oe = s + k + 1; k++; }
			} else {
				HB_CNS_FLUSH(); if (nf) break; os = oe = (uint64_t)-1;
				k += hb_bits_run(mP, k, (uint32_t)wl, 0);
			}
		}
#undef HB_CNS_FLUSH
		if (!nf) { occ.mms = occ.mme = (uint64_t)-1; if (oe > os && os != (uint64_t)-1) { occ.mms = os; occ.mme = oe; } }
	}
	*need_full = (int)hb_bcast((uint32_t)nf, 0);
	return rr;
}

// wcns_gen for a warp, called by every lane; S = the warp's shared-memory words.  The edit script, nec, C.need_full, C.ovf are lane 0's.
template <bool GRAPH> HB_HD uint64_t hb_cns_read_w(CnsCtx &C, uint64_t *S, uint32_t n_ov, uint32_t *srt, uint32_t *act_a, uint32_t *act_b, uint64_t *key)
{
	const int lane = hb_lane(); uint32_t n_ent = 0; uint64_t nec = 0;
	if (lane == 0) {
		for (uint32_t k = 0; k < n_ov; k++) {
			const CnsOv &z = C.ov[k];
			for (uint32_t i = 0; i < z.wn; i++) {
				if (hb_ualn_w(z.w[i])) continue;
				if (z.w[i].x_end >= z.w[i].x_start) {
					key[n_ent] = ((uint64_t)(uint32_t)z.w[i].x_start << 32) + n_ent;
					CnsEnt &p = C.ent[n_ent]; p.ov = k; p.wid = i; p.xoff = (uint32_t)z.w[i].x_start; p.yoff = (uint32_t)z.w[i].y_start; p.coff = 0;
					n_ent++;
				}
			}
		}
		hb_heapsort64(key, n_ent);
		int64_t k, i, t;
		for (k = 1, i = 0; k < (int64_t)n_ent; k++) {
			if ((key[k] >> 32) != (key[i] >> 32)) {
				if (k - i > 1) {
					for (t = i; t < k; t++) { const CnsEnt &cp = C.ent[(uint32_t)key[t]]; uint64_t m = (uint64_t)((int64_t)C.ov[cp.ov].w[cp.wid].x_end + 1); m <<= 32; m += (uint32_t)key[t]; key[t] = m; }
					hb_heapsort64(key + i, (uint32_t)(k - i));
				}
				i = k;
			}
		}
		for (uint32_t t2 = 0; t2 < n_ent; t2++) srt[t2] = (uint32_t)key[t2];
	}
	n_ent = hb_bcast(n_ent, 0);
	C.A.srt = srt; C.A.act = act_a; C.A.i = 0; C.A.srt_n = n_ent; C.A.act_n = 0; C.A.rr = C.A.ru = 0; C.A.mms = C.A.mme = (uint64_t)-1;
	C.B.srt = srt; C.B.act = act_b; C.B.i = 0; C.B.srt_n = n_ent; C.B.act_n = 0; C.B.rr = C.B.ru = 0; C.B.mms = C.B.mme = (uint64_t)-1;
	C.out_n = 0; C.has_win = 0; C.ax_start = C.ax_end = -1; C.ovf = 0; C.need_full = 0; C.b32_n = 0;
	hb_wsync();
	int64_t s = 0, e = HB_CNS_WL, rr = 0; if (e > C.ql) e = C.ql;
	for (; s < C.ql;) {
		uint32_t rn = 0;
		if (lane == 0) rn = hb_cns_iter(C, C.A, s, e, rr, 0);
		rn = hb_bcast(rn, 0);
		hb_wsync();
		int nf = 0;
		rr = hb_cns_vote_w<GRAPH>(C, S, rn, (uint64_t)s, (uint64_t)e, &nec, &nf);
		if (nf) { C.need_full = C.need_full ? C.need_full : 1; return nec; }
		s += HB_CNS_WL; e += HB_CNS_WL; if (e > C.ql) e = C.ql;
	}
	if (lane == 0) {
		if (C.B.mme > C.B.mms && C.B.mms != (uint64_t)-1) nec += hb_cns_anchor<GRAPH>(C, C.B.mms, C.B.mme, 0);
		if (!C.need_full) nec += hb_cns_anchor<GRAPH>(C, (uint64_t)C.ql, (uint64_t)C.ql, 1);
	}
	C.need_full = (int)hb_bcast((uint32_t)C.need_full, 0);
	return nec;
}
