// hb_eccns_full.cuh — the graph consensus of the window consensus (SURVEY.md §8 row a14, second half): cns_gen_full (ecovlp.cpp:1919).
//
// When the stretch between two anchors is longer than 6 columns, or its short variants have no majority, the reference builds a small DAG:
// backbone = the read's bases of the stretch (<= 256 per chunk) between a start and an end node (init_cns_g 630); every spanning window
// alignment is threaded through it run by run (extract_sub_cigar_cns 850 -> append_cns_g 791: matches walk the backbone (push_cns_c0 671),
// mismatches / insertions follow or create off-backbone nodes by base (push_cns_c1 771, trace_cns_bp 703, add_cns_arc_bp 602)), arc weights
// count the supporting alignments; refine_cns_g (1437) merges sibling nodes of equal base in topological order (merge_cns_g_in / _ou 1297 /
// 1364, gen_mm_cns_arc 1220, del_cns_g_nn 1264); gseq_cns_g (1488) takes the heaviest path; push_correct1_fhc (1798) turns the path into
// edit-script entries, and a deletion that follows inserted bases is re-aligned against the read (push_correct1_fhc_indel_exz 1618, banded
// global Myers with thresholds 31 / 63).  Node arcs are kept as the reference keeps them — per node one array, out-arcs first — because the
// iteration order decides ties.  One thread per read; the graph lives in a per-thread arena (CnsG); an arena that is too small is reported.
#pragma once
#include "hb_eccns.cuh"

#define HB_CNS_G_WL 256            // cns_g_wl, ecovlp.cpp:3309
#define HB_CNS_DEL_E 0x7fffffffu   // CNS_DEL_E, ecovlp.cpp:11
#define HB_CNS_DEL_V 0x1fffffffu   // CNS_DEL_V, ecovlp.cpp:13

struct CnsArc { uint32_t vf, sc; };  // cns_arc: v (31 bits) | f << 31, sc
struct CnsNode { uint32_t c, f, sc, off, n, nou, cap; }; // cns_t: base (2 bits), flag, score (29 bits); arc array = arc[off .. off + n), out-arcs [0, nou)
struct CnsG {
	CnsNode *nd; uint32_t n, ncap; CnsArc *arc; uint32_t arc_used, arc_cap;
	uint32_t si, ei, off, bn, bb0, bb1;
	uint32_t *q; uint32_t q_cap, q_front, q_count;            // kdq_t(uint32_t)
	uint32_t *b32; uint32_t b32_n, b32_cap;                   // asg32_v b32 of the graph path
	uint8_t *nseq; uint32_t *nseq_np; uint32_t nseq_cap;      // the locally corrected sequence of push_correct1_fhc_indel_exz: packed 2-bit + N positions
	MwEz ez;                                                  // aligner scratch (cal_exz_global)
	int ovf;
};
#define HB_ARC_V(a) ((a).vf & 0x7fffffffu)
#define HB_ARC_F(a) ((a).vf >> 31)
HB_HD void hb_arc_set_v(CnsArc &a, uint32_t v) { a.vf = (a.vf & 0x80000000u) | (v & 0x7fffffffu); }
HB_HD void hb_arc_set_f(CnsArc &a, uint32_t f) { a.vf = (a.vf & 0x7fffffffu) | (f << 31); }
HB_HD bool hb_g_del_arc(const CnsG &G, uint32_t v, uint32_t k) { return HB_ARC_V(G.arc[G.nd[v].off + k]) == HB_CNS_DEL_E; }
HB_HD bool hb_g_del_nn(const CnsG &G, uint32_t v) { return G.nd[v].sc == HB_CNS_DEL_V; }
#define HB_GA(G, v, k) ((G).arc[(G).nd[(v)].off + (k)])

// kv_pushp on a node's arc array (capacity doubles from 2; a grown array moves to the end of the arena)
HB_HD uint32_t hb_g_pushp(CnsG &G, uint32_t v)
{
	CnsNode &x = G.nd[v];
	if (x.n == x.cap) {
		const uint32_t nc = x.cap ? x.cap << 1 : 2;
		if (G.arc_used + nc > G.arc_cap) { G.ovf = 1; return 0xffffffffu; }
		for (uint32_t k = 0; k < x.n; k++) G.arc[G.arc_used + k] = G.arc[x.off + k];
		x.off = G.arc_used; G.arc_used += nc; x.cap = nc;
	}
	return x.n++;
}
// insert_cns_arc, ecovlp.cpp:519-535
HB_HD void hb_g_insert_arc(CnsG &G, uint32_t src, uint32_t des, uint32_t is_ou, uint32_t plus0)
{
	if (src >= G.n) { G.ovf = 1; return; }
	const uint32_t pi = hb_g_pushp(G, src); if (pi == 0xffffffffu) return;
	CnsNode &x = G.nd[src]; CnsArc p; p.vf = des & 0x7fffffffu; p.sc = plus0; G.arc[x.off + pi] = p;
	if (is_ou) {
		x.nou++;
		if (x.nou < x.n) { const CnsArc t = G.arc[x.off + x.nou - 1]; G.arc[x.off + x.nou - 1] = G.arc[x.off + pi]; G.arc[x.off + pi] = t; }
	}
}
// insert_cns_node, ecovlp.cpp:537-552
HB_HD uint32_t hb_g_insert_node(CnsG &G)
{
	if (G.n >= G.ncap) { G.ovf = 1; return 0; }
	CnsNode &p = G.nd[G.n++]; p.n = p.nou = 0; p.c = p.f = p.sc = 0; p.cap = 0; p.off = 0;
	return G.n - 1;
}
// add_cns_arc, ecovlp.cpp:554-571
HB_HD uint32_t hb_g_add_arc(CnsG &G, uint32_t src, uint32_t des, uint32_t is_ou, uint32_t plus)
{
	const CnsNode &x = G.nd[src]; uint32_t k, s, e;
	if (is_ou) { s = 0; e = x.nou; } else { s = x.nou; e = x.n; }
	for (k = s; k < e; k++) if (HB_ARC_V(G.arc[x.off + k]) == des) { G.arc[x.off + k].sc += plus; break; }
	return k < e ? 1 : 0;
}
// get_cns_arc_bp, ecovlp.cpp:582-600
HB_HD uint32_t hb_g_get_arc_bp(const CnsG &G, uint32_t src, uint32_t bp, uint32_t is_ou, uint32_t av_bp)
{
	const CnsNode &x = G.nd[src]; uint32_t k, s, e;
	if (is_ou) { s = 0; e = x.nou; } else { s = x.nou; e = x.n; }
	for (k = s; k < e; k++) {
		const uint32_t v = HB_ARC_V(G.arc[x.off + k]);
		if (v == 0 || v == 1) continue;
		if (av_bp && v >= G.bb0 && v < G.bb1) continue;
		if (v < G.n && G.nd[v].c == bp) return k;
	}
	return 0xffffffffu;
}
// add_cns_arc_bp, ecovlp.cpp:602-628
HB_HD uint32_t hb_g_add_arc_bp(CnsG &G, uint32_t src, uint32_t bp, uint32_t plus0, uint32_t av_bp)
{
	uint32_t rr = hb_g_get_arc_bp(G, src, bp, 1, av_bp), des;
	if (rr != 0xffffffffu) {
		des = HB_ARC_V(HB_GA(G, src, rr)); G.nd[des].sc++; HB_GA(G, src, rr).sc += plus0;
		hb_g_add_arc(G, des, src, 0, plus0);
		return des;
	}
	des = hb_g_insert_node(G); if (G.ovf) return src;
	G.nd[des].sc++; G.nd[des].c = bp & 3; // the node keeps two bits of the code (an N, code 5, becomes 1)
	hb_g_insert_arc(G, src, des, 1, plus0); hb_g_insert_arc(G, des, src, 0, plus0);
	return des;
}
// init_cns_g, ecovlp.cpp:630-668: backbone of the read's bases [qoff, qoff + sl)
HB_HD void hb_g_init(CnsG &G, const RdView &q, int64_t qoff, uint32_t sl)
{
	G.n = 0; G.arc_used = 0; G.si = 0; G.ei = 1; G.off = 2; G.ovf = 0;
	if (sl + 2 > G.ncap) { G.ovf = 1; return; }
	hb_g_insert_node(G); hb_g_insert_node(G); G.bb0 = G.n;
	for (uint32_t k = 0; k < sl; k++) {
		const uint32_t id = hb_g_insert_node(G); const int b = q.at(qoff + k);
		G.nd[id].c = (uint32_t)(b == 4 ? 5 : b) & 3; G.nd[id].sc = 1; // seq_nt6_table: N -> 5, two bits kept
		if (k + 1 < sl) hb_g_insert_arc(G, k + G.off, k + 1 + G.off, 1, 1);
		if (k > 0) hb_g_insert_arc(G, k + G.off, k - 1 + G.off, 0, 1);
	}
	if (sl) {
		hb_g_insert_arc(G, G.si, 0 + G.off, 1, 1); hb_g_insert_arc(G, 0 + G.off, G.si, 0, 1);
		hb_g_insert_arc(G, sl - 1 + G.off, G.ei, 1, 1); hb_g_insert_arc(G, G.ei, sl - 1 + G.off, 0, 1);
	} else { hb_g_insert_arc(G, G.si, G.ei, 1, 1); hb_g_insert_arc(G, G.ei, G.si, 0, 1); }
	G.bn = G.n; G.bb1 = G.n;
}
// push_cns_c0, ecovlp.cpp:671-701: a match run walks the backbone nodes [s, e)
HB_HD uint32_t hb_g_push_c0(CnsG &G, uint64_t s0, uint64_t s, uint64_t e, uint32_t plus0)
{
	if (s > e) return (uint32_t)s0;
	uint32_t k, re;
	if (!hb_g_add_arc(G, (uint32_t)s0, (uint32_t)s, 1, plus0)) { hb_g_insert_arc(G, (uint32_t)s0, (uint32_t)s, 1, plus0); hb_g_insert_arc(G, (uint32_t)s, (uint32_t)s0, 0, plus0); }
	else hb_g_add_arc(G, (uint32_t)s, (uint32_t)s0, 0, plus0);
	if (s >= G.n) { G.ovf = 1; return (uint32_t)s0; }
	G.nd[s].sc++; re = (uint32_t)s;
	for (k = (uint32_t)s + 1; k < e; k++) { hb_g_add_arc(G, k - 1, k, 1, 1); hb_g_add_arc(G, k, k - 1, 0, 1); G.nd[k].sc++; re = k; }
	return re;
}
// trace_cns_bp, ecovlp.cpp:703-768: follow existing off-backbone nodes that spell the target bases tb[0..tl) from s0 (breadth first, first match wins)
HB_HD uint32_t hb_g_trace_bp(CnsG &G, uint64_t s0, const RdView &T, int64_t toff, uint64_t tl, uint32_t plus0, uint32_t *rn, uint64_t max_trace, uint32_t av_bp)
{
	*rn = (uint32_t)s0;
	if (tl <= 0) return 0;
	uint32_t k, i, e, m, bp, nm, bi, bn0, src, des, ff = 0; G.b32_n = 0;
	if (G.b32_cap < 4) { G.ovf = 1; return 0; }
	G.b32[G.b32_n++] = (uint32_t)s0; G.b32[G.b32_n++] = 0xffffffffu; nm = 2;
	for (i = 0; i < tl && !ff; i++) {
		const int b = T.at(toff + i); bp = (uint32_t)(b == 4 ? 5 : b); bn0 = G.b32_n;
		for (bi = bn0 - nm; bi < bn0; bi += 2) {
			m = G.b32[bi]; e = G.nd[m].nou;
			for (k = 0; k < e; k++) {
				const uint32_t v = HB_ARC_V(HB_GA(G, m, k));
				if (v == 0 || v == 1) continue;
				if (av_bp && v >= G.bb0 && v < G.bb1) continue;
				if (G.nd[v].c == bp) {
					if (G.b32_n + 2 > G.b32_cap) { G.ovf = 1; return 0; }
					G.b32[G.b32_n++] = v; G.b32[G.b32_n++] = bi;
					if ((i + 1) == tl || G.b32_n > max_trace) { ff = 1; break; }
				}
			}
			if (ff) break;
		}
		if (G.b32_n <= bn0) break; else nm = G.b32_n - bn0;
	}
	if (i > 0 && nm > 0) {
		*rn = G.b32[G.b32_n - nm];
		for (bi = G.b32_n - nm; G.b32[bi + 1] != 0xffffffffu; bi = G.b32[bi + 1]) {
			des = G.b32[bi]; src = G.b32[G.b32[bi + 1]]; bp = src != s0 ? 1 : plus0;
			hb_g_add_arc(G, src, des, 1, bp); hb_g_add_arc(G, des, src, 0, bp);
			G.nd[des].sc++;
		}
	} else i = 0;
	return i;
}
// push_cns_c1, ecovlp.cpp:771-789
HB_HD uint32_t hb_g_push_c1(CnsG &G, uint64_t s0, const RdView &T, int64_t toff, uint64_t tl, uint32_t plus0, uint64_t max_trace)
{
	if (tl <= 0) return (uint32_t)s0;
	uint32_t rr = plus0, k, re = (uint32_t)s0;
	k = hb_g_trace_bp(G, s0, T, toff, tl, plus0, &re, max_trace, 1);
	if (k > 0) rr = 1;
	for (; k < tl && !G.ovf; k++) { const int b = T.at(toff + k); re = hb_g_add_arc_bp(G, re, (uint32_t)(b == 4 ? 5 : b), rr, 1); rr = 1; }
	return re;
}
// append_cns_g, ecovlp.cpp:791-821
HB_HD uint64_t hb_g_append(CnsG &G, const RdView &T, int64_t toff, uint64_t tl, uint64_t qs, uint64_t qe, uint64_t cp, uint64_t cl, uint64_t pe, uint64_t max_trace, int64_t insert_pos)
{
	uint64_t s0 = pe, plus0 = 1, ns = qs + G.off, ne = qe + G.off;
	if (pe == (uint64_t)-1) s0 = qs > 0 ? qs - 1 + G.off : 0;
	if (cp == 0) {
		if (cl == 0 && qs == qe && (int64_t)qe == insert_pos) { s0 = 0; ns = ne = 1; plus0 = 1; }
		return hb_g_push_c0(G, s0, ns, ne, (uint32_t)plus0);
	} else if (cp == 1 || cp == 2) return hb_g_push_c1(G, s0, T, toff, tl, (uint32_t)plus0, max_trace);
	return s0;
}
// extract_sub_cigar_cns, ecovlp.cpp:850-1053: thread one window alignment through the graph of the stretch [iws, iwe)
HB_HD void hb_cns_sub_cns(CnsCtx &C, CnsG &G, CnsEnt &p, int64_t s, int64_t e, int64_t iws, int64_t iwe, int64_t s_end, uint64_t max_trace)
{
	const CnsOv &z = C.ov[p.ov]; const hb_wl_t &w = z.w[p.wid];
	int64_t xk = p.xoff, yk = p.yoff, ck = p.coff, os, oe, ots, ote, ol, ii0, ii1; const int64_t insert_pos = iws == iwe ? 0 : -1; uint64_t pe = (uint64_t)-1;
	const int64_t s0 = w.x_start, e0 = (int64_t)w.x_end + 1;
	if (s < s0) s = s0; if (e > e0) e = e0;
	if (s > e) return;
	os = s > s0 ? s : s0; oe = e < e0 ? e : e0;
	if (oe < os) return;
	const uint16_t *cg = C.pool + w.cidx; const int64_t cn = w.clen;
	if (!cn) return;
	uint32_t op; int64_t ws, we, wts, wte, ovlp;
	if (ck < 0 || ck > cn) { ck = 0; xk = w.x_start; yk = w.y_start; }
	while (ck > 0 && xk >= s) { --ck; op = cg[ck] >> 14; if (op != 2) xk -= cg[ck] & 0x3fff; if (op != 3) yk -= cg[ck] & 0x3fff; }
	if (s_end == 0 && s == iws) s_end = 0; else s_end = 1;
	ii0 = ii1 = -1;
	const RdView T = hb_rd_view(C.R, z.y_id, z.rev);
	while (ck < cn && xk < e) {
		ws = xk; wts = yk; op = cg[ck] >> 14; ol = cg[ck] & 0x3fff;
		for (ck++; ck < cn && op == (uint32_t)(cg[ck] >> 14); ck++) ol += cg[ck] & 0x3fff;
		if (op != 2) xk += ol; if (op != 3) yk += ol;
		we = xk; wte = yk;
		os = s > ws ? s : ws; oe = e < we ? e : we; ovlp = oe > os ? oe - os : 0;
		if (s == e) { if (op != 0 || ws >= s || we <= e || e != iwe || s != iws) continue; }
		else { if (op != 2) { if (!ovlp) continue; } else { if (ws < s || ws >= e) continue; } }
		if (s_end == 0 && op == 2 && ws == s) continue;
		if (op < 2) { ots = os - ws + wts; ote = oe - ws + wts; } else { ots = wts; ote = wte; }
		if (ii0 == -1) ii0 = os;
		ii1 = oe;
		if (op != 2) ol = oe - os;
		pe = hb_g_append(G, T, ots, (uint64_t)(op != 0 ? ote - ots : 0), (uint64_t)(os - iws), (uint64_t)(oe - iws), op, (uint64_t)ol, pe, max_trace, insert_pos);
		if (G.ovf) return;
	}
	while (ck < cn && xk <= e) {
		ws = xk; wts = yk; op = cg[ck] >> 14; ol = cg[ck] & 0x3fff;
		if (op != 2) break;
		for (ck++; ck < cn && op == (uint32_t)(cg[ck] >> 14); ck++) ol += cg[ck] & 0x3fff;
		yk += ol; we = xk; wte = yk;
		if (ws >= s && ws <= e) {
			ots = wts; ote = wte;
			if (ii0 == -1) ii0 = ws;
			ii1 = we;
			pe = hb_g_append(G, T, ots, (uint64_t)(ote - ots), (uint64_t)(ws - iws), (uint64_t)(we - iws), op, (uint64_t)ol, pe, max_trace, insert_pos);
			if (G.ovf) return;
		}
	}
	if (ii1 == -1) return; // (the cursor is not advanced on this exit, as in the reference)
	uint64_t ae = ii1 == iwe ? 1 : (uint64_t)(ii1 + G.off - iws);
	if (pe == (uint64_t)-1) pe = 0;
	if (pe != ae) {
		if (!hb_g_add_arc(G, (uint32_t)pe, (uint32_t)ae, 1, 1)) { hb_g_insert_arc(G, (uint32_t)pe, (uint32_t)ae, 1, 1); hb_g_insert_arc(G, (uint32_t)ae, (uint32_t)pe, 0, 1); }
		else hb_g_add_arc(G, (uint32_t)ae, (uint32_t)pe, 0, 1);
	}
	p.xoff = (uint32_t)xk; p.yoff = (uint32_t)yk; p.coff = (int32_t)ck;
}
// gen_mm_cns_arc, ecovlp.cpp:1220-1262
HB_HD void hb_g_mm_arc(CnsG &G, uint32_t src, uint32_t des, uint32_t sc, uint32_t f)
{
	uint32_t vk, wk;
	for (vk = 0; vk < G.nd[src].nou; vk++) {
		if (HB_ARC_V(HB_GA(G, src, vk)) != des) continue; // (a deleted arc never equals des)
		hb_arc_set_f(HB_GA(G, src, vk), f); HB_GA(G, src, vk).sc += sc;
		for (wk = G.nd[des].nou; wk < G.nd[des].n; wk++) {
			if (HB_ARC_V(HB_GA(G, des, wk)) != src) continue;
			hb_arc_set_f(HB_GA(G, des, wk), f); HB_GA(G, des, wk).sc += sc; break;
		}
		return;
	}
	uint32_t pi = hb_g_pushp(G, src); if (pi == 0xffffffffu) return;
	{ CnsArc a; a.vf = (des & 0x7fffffffu) | (f << 31); a.sc = sc; HB_GA(G, src, pi) = a; }
	CnsNode &x = G.nd[src]; x.nou++;
	if (x.nou < x.n) { const CnsArc t = G.arc[x.off + x.nou - 1]; G.arc[x.off + x.nou - 1] = G.arc[x.off + pi]; G.arc[x.off + pi] = t; }
	pi = hb_g_pushp(G, des); if (pi == 0xffffffffu) return;
	{ CnsArc a; a.vf = (src & 0x7fffffffu) | (f << 31); a.sc = sc; HB_GA(G, des, pi) = a; }
}
// del_cns_g_nn, ecovlp.cpp:1264-1295
HB_HD void hb_g_del_node(CnsG &G, uint32_t v)
{
	uint32_t w, vk, wk;
	for (vk = 0; vk < G.nd[v].nou; vk++) {
		if (hb_g_del_arc(G, v, vk)) continue;
		w = HB_ARC_V(HB_GA(G, v, vk)); hb_arc_set_v(HB_GA(G, v, vk), HB_CNS_DEL_E);
		for (wk = G.nd[w].nou; wk < G.nd[w].n; wk++) { if (HB_ARC_V(HB_GA(G, w, wk)) != v) continue; hb_arc_set_v(HB_GA(G, w, wk), HB_CNS_DEL_E); break; }
	}
	for (vk = G.nd[v].nou; vk < G.nd[v].n; vk++) {
		if (hb_g_del_arc(G, v, vk)) continue;
		w = HB_ARC_V(HB_GA(G, v, vk)); hb_arc_set_v(HB_GA(G, v, vk), HB_CNS_DEL_E);
		for (wk = 0; wk < G.nd[w].nou; wk++) { if (HB_ARC_V(HB_GA(G, w, wk)) != v) continue; hb_arc_set_v(HB_GA(G, w, wk), HB_CNS_DEL_E); break; }
	}
	G.nd[v].n = G.nd[v].nou = 0; G.nd[v].c = G.nd[v].f = 0; G.nd[v].sc = HB_CNS_DEL_V;
}
// merge_cns_g_in / merge_cns_g_ou, ecovlp.cpp:1297-1435: in-neighbours (out-neighbours) of v with the same base and v as their only
// successor (predecessor) collapse into the first of them; repeated on the merged node
HB_HD void hb_g_merge(CnsG &G, uint32_t v0, int is_in)
{
	uint32_t v, bp, vk, wk, wka, w, wn, nn, mn, wh, mk0, mk1;
	G.b32_n = 0; G.b32[G.b32_n++] = v0;
	while (G.b32_n && !G.ovf) {
		v = G.b32[--G.b32_n];
		if (hb_g_del_nn(G, v)) continue;
		for (bp = 0; bp < 4; bp++) {
			nn = wh = 0; mn = mk0 = mk1 = wka = 0xffffffffu;
			const uint32_t vs = is_in ? G.nd[v].nou : 0;
			for (vk = vs; vk < (is_in ? G.nd[v].n : G.nd[v].nou); vk++) {
				if (hb_g_del_arc(G, v, vk)) continue;
				w = HB_ARC_V(HB_GA(G, v, vk));
				if (G.nd[w].c != bp) continue;
				if (w == G.si || w == G.ei) continue;
				if (is_in) { for (wk = wn = 0; wk < G.nd[w].nou; wk++) { if (hb_g_del_arc(G, w, wk)) continue; wn++; wka = wk; if (wn > 1) break; } }
				else { for (wk = G.nd[w].nou, wn = 0; wk < G.nd[w].n; wk++) { if (hb_g_del_arc(G, w, wk)) continue; wn++; wka = wk; if (wn > 1) break; } }
				if (wn != 1) continue;
				if (nn == 0) { mn = w; mk0 = vk; mk1 = wka; wh = HB_GA(G, v, vk).sc; }
				else wh += HB_GA(G, w, wka).sc;
				if (nn > 0) {
					if (is_in) { for (wk = G.nd[w].nou; wk < G.nd[w].n; wk++) { if (hb_g_del_arc(G, w, wk)) continue; const CnsArc a = HB_GA(G, w, wk); hb_g_mm_arc(G, HB_ARC_V(a), mn, a.sc, HB_ARC_F(a)); } }
					else { for (wk = 0; wk < G.nd[w].nou; wk++) { if (hb_g_del_arc(G, w, wk)) continue; const CnsArc a = HB_GA(G, w, wk); hb_g_mm_arc(G, mn, HB_ARC_V(a), a.sc, HB_ARC_F(a)); } }
					hb_g_del_node(G, w);
				}
				nn++;
			}
			if (nn) {
				HB_GA(G, v, mk0).sc = wh; HB_GA(G, mn, mk1).sc = wh;
				if (G.b32_n >= G.b32_cap) { G.ovf = 1; return; }
				G.b32[G.b32_n++] = mn;
			}
		}
	}
}
HB_HD void hb_g_q_push(CnsG &G, uint32_t v) { if (G.q_count >= G.q_cap) { G.ovf = 1; return; } G.q[(G.q_front + G.q_count) % G.q_cap] = v; G.q_count++; }
HB_HD bool hb_g_q_shift(CnsG &G, uint32_t *v) { if (!G.q_count) return false; *v = G.q[G.q_front]; G.q_front = (G.q_front + 1) % G.q_cap; G.q_count--; return true; }
// refine_cns_g, ecovlp.cpp:1437-1486
HB_HD void hb_g_refine(CnsG &G)
{
	uint32_t v, w, vk, wk;
	G.q_front = G.q_count = 0; hb_g_q_push(G, G.si);
	while (!G.ovf && hb_g_q_shift(G, &v)) {
		if (hb_g_del_nn(G, v)) continue;
		hb_g_merge(G, v, 1); hb_g_merge(G, v, 0);
		for (vk = 0; vk < G.nd[v].nou; vk++) {
			if (hb_g_del_arc(G, v, vk)) continue;
			if (HB_ARC_F(HB_GA(G, v, vk)) == 0) continue;
			hb_arc_set_f(HB_GA(G, v, vk), 1); w = HB_ARC_V(HB_GA(G, v, vk));
			for (wk = G.nd[w].nou; wk < G.nd[w].n; wk++) { if (HB_ARC_V(HB_GA(G, w, wk)) != v) continue; hb_arc_set_f(HB_GA(G, w, wk), 1); break; }
		}
		G.nd[v].f = 1;
		for (vk = 0; vk < G.nd[v].nou; vk++) {
			if (hb_g_del_arc(G, v, vk)) continue;
			w = HB_ARC_V(HB_GA(G, v, vk));
			for (wk = G.nd[w].nou; wk < G.nd[w].n; wk++) {
				if (hb_g_del_arc(G, w, wk)) continue;
				if (HB_ARC_F(HB_GA(G, w, wk))) continue;
				if (G.nd[HB_ARC_V(HB_GA(G, w, wk))].f) continue;
				break;
			}
			if (wk >= G.nd[w].n) hb_g_q_push(G, w);
		}
	}
}
// gseq_cns_g, ecovlp.cpp:1488-1559: heaviest path from the start to the end node -> G.b32[0 .. b32_n)
HB_HD void hb_g_seq(CnsG &G, uint32_t bl)
{
	uint32_t v, vk, w, mme, mmn, mmk, mmw, sw; uint32_t *ii = G.b32; const uint32_t bs = G.off, be = bl + G.off;
	if (G.n > G.b32_cap) { G.ovf = 1; return; }
	G.b32_n = 0;
	for (v = 0; v < G.n; v++) {
		ii[v] = 0;
		if (hb_g_del_nn(G, v)) continue;
		G.nd[v].sc = 0; G.nd[v].f = 0;
		for (vk = G.nd[v].nou; vk < G.nd[v].n; vk++) { if (hb_g_del_arc(G, v, vk)) continue; G.nd[v].sc++; }
	}
	G.q_front = G.q_count = 0; hb_g_q_push(G, G.si);
	while (!G.ovf && hb_g_q_shift(G, &v)) {
		if (hb_g_del_nn(G, v)) continue;
		for (vk = G.nd[v].nou, mme = mmn = mmw = 0, mmk = 0xffffffffu; vk < G.nd[v].n; vk++) {
			if (hb_g_del_arc(G, v, vk)) continue;
			w = HB_ARC_V(HB_GA(G, v, vk)); sw = (w >= bs && w < be) ? 1 : 0; const uint32_t asc = HB_GA(G, v, vk).sc;
			if (mmk == 0xffffffffu || asc > mme || (asc == mme && ii[w] > mmn) || (asc == mme && ii[w] == mmn && sw == 1 && mmw == 0)) { mmk = vk; mme = asc; mmn = ii[w]; mmw = sw; }
		}
		ii[v] = mme + mmn; G.nd[v].f = 1;
		G.nd[v].sc = mmk != 0xffffffffu ? HB_ARC_V(HB_GA(G, v, mmk)) : v;
		for (vk = 0; vk < G.nd[v].nou; vk++) {
			if (hb_g_del_arc(G, v, vk)) continue;
			w = HB_ARC_V(HB_GA(G, v, vk));
			G.nd[w].sc = (G.nd[w].sc - 1) & 0x1fffffffu; // (29-bit field)
			if (G.nd[w].sc == 0) hb_g_q_push(G, w);
		}
	}
	uint32_t guard = 0;
	for (v = G.nd[G.ei].sc, G.b32_n = 0; v != G.si; v = G.nd[v].sc) { if (v >= G.n || ++guard > G.n) { G.ovf = 1; return; } G.b32[G.b32_n++] = v; }
	for (vk = 0; vk < (G.b32_n >> 1); vk++) { v = G.b32[vk]; G.b32[vk] = G.b32[G.b32_n - vk - 1]; G.b32[G.b32_n - vk - 1] = v; }
}

// ---- the path back into the edit script ------------------------------------------------------------------------------------------------
HB_HD uint32_t hb_nt6(int b) { return (uint32_t)(b == 4 ? 5 : b); } // seq_nt6_table on a decoded base (Process_Read.cpp:12): N -> 5
// push_correct1_fhc_indel_exz, ecovlp.cpp:1618-1796 (c0 == 3): the deletion [ok0, ok0 + cl0) of the stretch follows edits since the last match run of
// this call (script entries [sc0, n)); unless those are all deletions, the old and the locally corrected sequence are re-aligned and the shorter script kept
HB_HD uint64_t hb_cns_indel_exz(CnsCtx &C, CnsG &G, int64_t sc0, int64_t qoff, uint64_t gbeg, int64_t cl0, int64_t ok0)
{
	int64_t ck = C.out_n, k, ok = 0, nk = 0, cn, cn0, nl, ol, diff, diff0, ml, ml0, e0 = 0; uint32_t on, f = 0, nec = 0, op;
	const uint32_t c0 = 3;
	ok += cl0; e0 += cl0;
	for (ck--; ck >= sc0; ck--) {
		op = C.out[ck] >> 14;
		if (!op) break;
		if (op == 2 || op == 3) on = C.out[ck] & 0xfff; else if (op == 1) on = C.out[ck] & 0x3ff; else on = C.out[ck] & 0x3fff;
		if (op != 2) ok += on; if (op != 3) nk += on; if (op != 0) e0 += on;
		if (c0 != op) f = 1;
	}
	cn0 = ck + 1; cn = C.out_n;
	if (!f || !ok || !nk) {
		for (k = 0, ck = ok0 + (int64_t)gbeg; k < cl0; k++, ck++) { hb_sc_push(C, c0, G.nd[ck].c, HB_SC_NONE, 1, C.out_n > 0 ? 1 : 0); nec++; }
		return nec;
	}
	int64_t wo0 = 0, wo1 = 0, wn0 = 0, wn1 = 0; ScRun r;
	ok0 += cl0; ok0 -= ok;
	if (ok0 < 0 || (uint64_t)nk + 8 > G.nseq_cap) { G.ovf = 1; return nec; }
	const int64_t ooff = qoff + ok0; // oseq = ostr + ok0
	ol = ok; nl = nk; ck = cn0; ok = nk = 0;
	uint32_t n_np = 0;
	for (k = 0; k < (nl + 3) / 4 + 1; k++) G.nseq[k] = 0;
	auto put = [&](int64_t pos, int b) { if (b == 4) { G.nseq_np[n_np++] = (uint32_t)pos; b = 0; } G.nseq[pos >> 2] |= (uint8_t)(b << ((3 - (pos & 3)) << 1)); };
	while (ck < cn) {
		wo0 = ok; wn0 = nk;
		ck = hb_sc_pop(C.out, (uint32_t)cn, (uint32_t)ck, &r);
		if (r.op != 2) ok += r.len; if (r.op != 3) nk += r.len;
		wo1 = ok; wn1 = nk;
		if (r.op == 0) for (k = 0; k < wo1 - wo0; k++) put(wn0 + k, C.q.at(ooff + wo0 + k));
		else if (r.op == 1 || r.op == 2) for (k = wn0; k < wn1; k++) put(k, (int)r.bt);
	}
	RdView NS; NS.p = G.nseq; NS.npos = G.nseq_np; NS.nn = n_np; NS.len = (uint32_t)nl; NS.rev = 0;
	if (nl == ol && nl == 1) {
		C.out_n = (uint32_t)cn0;
		const int ob = C.q.at(ooff), nb = NS.at(0);
		if (ob == nb) hb_sc_push(C, 0, HB_SC_NONE, HB_SC_NONE, 1, C.out_n > 0 ? 1 : 0);
		else { hb_sc_push(C, 1, hb_nt6(ob), hb_nt6(nb), 1, C.out_n > 0 ? 1 : 0); nec++; }
		return nec;
	}
	ml = ol > nl ? ol : nl; f = 0;
	MwEz &ez = G.ez;
	diff = 31; if (diff > ml) diff = ml; diff0 = diff; ez.err = INT32_MAX; ez.ovf = 0;
	hb_mw_align(0, NS, 0, (int32_t)nl, C.q, ooff, (int32_t)ol, (int32_t)diff, 0, ez);
	if (ez.ovf) { G.ovf = 1; return nec; }
	if (ez.err <= ez.thre) f = 1;
	if (!f) {
		diff = 63; if (diff > ml) diff = ml;
		if (diff > diff0) {
			diff0 = diff; ez.err = INT32_MAX;
			hb_mw_align(0, NS, 0, (int32_t)nl, C.q, ooff, (int32_t)ol, (int32_t)diff, 0, ez);
			if (ez.ovf) { G.ovf = 1; return nec; }
			if (ez.err <= ez.thre) f = 1;
		}
	}
	if (f && ez.err < e0) {
		C.out_n = (uint32_t)cn0; const int32_t ecn = ez.cn; ok = nk = 0; uint32_t c, cl;
		for (uint32_t ci = 0; ci < (uint32_t)ecn;) {
			wo0 = ok; wn0 = nk;
			ci = hb_cg_pop(ez.cig, (uint32_t)ecn, ci, &c, &cl);
			if (c != 2) ok += cl; if (c != 3) nk += cl;
			if (c == 0) hb_sc_push(C, 0, HB_SC_NONE, HB_SC_NONE, cl, C.out_n > 0 ? 1 : 0);
			else if (c == 1) for (k = 0; k < (int64_t)cl; k++) { hb_sc_push(C, 1, hb_nt6(C.q.at(ooff + wo0 + k)), hb_nt6(NS.at(wn0 + k)), 1, C.out_n > 0 ? 1 : 0); nec++; }
			else if (c == 2) for (k = 0; k < (int64_t)cl; k++) { hb_sc_push(C, 2, HB_SC_NONE, hb_nt6(NS.at(wn0 + k)), 1, C.out_n > 0 ? 1 : 0); nec++; }
			else for (k = 0; k < (int64_t)cl; k++) { hb_sc_push(C, 3, hb_nt6(C.q.at(ooff + wo0 + k)), HB_SC_NONE, 1, C.out_n > 0 ? 1 : 0); nec++; }
		}
	} else if (ml < e0) {
		C.out_n = (uint32_t)cn0; ml0 = ol < nl ? ol : nl;
		for (k = 0; k < ml0; k++) { hb_sc_push(C, 1, hb_nt6(C.q.at(ooff + k)), hb_nt6(NS.at(k)), 1, C.out_n > 0 ? 1 : 0); nec++; }
		if (ol > ml0) for (k = ml0; k < ol; k++) { hb_sc_push(C, 3, hb_nt6(C.q.at(ooff + k)), HB_SC_NONE, 1, C.out_n > 0 ? 1 : 0); nec++; }
		else if (nl > ml0) for (k = ml0; k < nl; k++) { hb_sc_push(C, 2, HB_SC_NONE, hb_nt6(NS.at(k)), 1, C.out_n > 0 ? 1 : 0); nec++; }
	} else {
		for (k = 0, ck = ok0 + (int64_t)gbeg; k < cl0; k++, ck++) { hb_sc_push(C, c0, G.nd[ck].c, HB_SC_NONE, 1, C.out_n > 0 ? 1 : 0); nec++; }
	}
	return nec;
}
// push_correct1_fhc, ecovlp.cpp:1798-1861: rc = the path (G.b32), bl = length of the stretch, qoff = its start on the read
HB_HD uint64_t hb_cns_push1(CnsCtx &C, CnsG &G, int64_t qoff, uint32_t bl)
{
	uint64_t nec = 0; uint32_t k, l, i, ff, sl, sk; const uint32_t bs = G.off, be = bl + G.off; uint32_t bend = G.off, is_i = 0; const int64_t sc0 = C.out_n;
	const uint32_t *rc = G.b32; const uint32_t rn = G.b32_n;
	if (rn) {
		for (k = 1, l = 0; k <= rn; ++k) {
			ff = 0; sl = sk = 0;
			if (k == rn) { if (l < rn) sl = (rc[l] >= bs && rc[l] < be) ? 1 : 0; ff = 1; }
			else {
				sl = (rc[l] >= bs && rc[l] < be) ? 1 : 0; sk = (rc[k] >= bs && rc[k] < be) ? 1 : 0;
				if (sl != sk) ff = 1; else if (sl == 1 && (rc[k] - rc[l]) != (k - l)) ff = 1;
			}
			if (!ff) continue;
			if (sl) {
				if (rc[l] > bend) {
					if (is_i) nec += hb_cns_indel_exz(C, G, sc0, qoff, G.off, (int64_t)rc[l] - bend, (int64_t)bend - G.off);
					else for (i = bend; i < rc[l]; i++) { hb_sc_push(C, 3, G.nd[i].c, HB_SC_NONE, 1, C.out_n > 0 ? 1 : 0); nec++; }
					if (G.ovf) return nec;
				}
				hb_sc_push(C, 0, HB_SC_NONE, HB_SC_NONE, rc[k - 1] + 1 - rc[l], C.out_n > 0 ? 1 : 0);
				bend = rc[k - 1] + 1; is_i = 0;
			} else {
				for (i = l; i < k; i++) { hb_sc_push(C, 2, HB_SC_NONE, G.nd[rc[i]].c, 1, C.out_n > 0 ? 1 : 0); nec++; }
				is_i = 1;
			}
			l = k;
		}
	}
	if (be > bend) {
		if (is_i) nec += hb_cns_indel_exz(C, G, sc0, qoff, G.off, (int64_t)be - bend, (int64_t)bend - G.off);
		else for (i = bend; i < be; i++) { hb_sc_push(C, 3, G.nd[i].c, HB_SC_NONE, 1, C.out_n > 0 ? 1 : 0); nec++; }
	}
	return nec;
}
// cns_gen_full0, ecovlp.cpp:1864-1917
HB_HD uint64_t hb_cns_full0(CnsCtx &C, CnsG &G, int64_t s, int64_t e, int64_t s_end)
{
	hb_g_init(G, C.q, s, (uint32_t)(e - s));
	if (G.ovf) return 0;
	CnsIt &idx = C.B; G.b32_n = 0;
	const uint32_t id_n = hb_cns_iter(C, idx, s, e, idx.rr, s == e ? 1 : 0);
	idx.rr = 0;
	for (uint32_t k = 0; k < id_n; k++) {
		CnsEnt &p = C.ent[idx.act[k]]; const hb_wl_t &w = C.ov[p.ov].w[p.wid];
		const int64_t q0 = w.x_start, q1 = (int64_t)w.x_end + 1;
		if (q1 <= e) idx.rr = 1;
		const int64_t os = q0 > s ? q0 : s, oe = q1 < e ? q1 : e;
		if (oe > os || (s == e && s > q0 && s < q1)) { hb_cns_sub_cns(C, G, p, os, oe, s, e, s_end, (uint64_t)C.ql); if (G.ovf) return 0; }
	}
	hb_g_refine(G); if (G.ovf) return 0;
	hb_g_seq(G, (uint32_t)(e - s)); if (G.ovf) return 0;
	return hb_cns_push1(C, G, s, (uint32_t)(e - s));
}
// cns_gen_full, ecovlp.cpp:1919-1936: chunks of cns_g_wl columns
HB_HD uint64_t hb_cns_full(CnsCtx &C, CnsG &G, int64_t s0, int64_t e0)
{
	uint64_t nec = 0;
	if (e0 - s0 <= HB_CNS_G_WL) return hb_cns_full0(C, G, s0, e0, 1);
	int64_t s = s0, e = s0 + HB_CNS_G_WL; if (e > e0) e = e0;
	for (; s < e0 && !G.ovf;) { nec += hb_cns_full0(C, G, s, e, s == s0 ? 1 : 0); s += HB_CNS_G_WL; e += HB_CNS_G_WL; if (e > e0) e = e0; }
	return nec;
}
HB_HD_NI uint64_t hb_cns_full_(CnsCtx &C, int64_t s0, int64_t e0)
{
	const uint64_t nec = hb_cns_full(C, *C.g, s0, e0);
	if (C.g->ovf) C.need_full = 2;
	return nec;
}
