// Phasing paths of the bundles (bundle_base::build_phase_set, rnacore/bundle_base.cc:338-418): every bridged fragment and
// every hit outside a paired fragment contributes the exon-coordinate list [lpos(vertex of its start), intron chain ...,
// rpos(vertex of its end)] when that list is non-decreasing; phase_set (rnacore/phase_set.h) counts equal lists.
//
// Elements of bundle b live at E_off[b] = frg_off[b] + hit_off[b]: first its fragments, then its hits.  Pass 0 decides and
// measures, a device-wide scan places the coordinates, pass 1 writes them, then equal lists are merged in a per-bundle
// open-addressing table (the chain-set table of k_evidence.h) and the distinct ones are compacted in element order.  The
// fetches order them (phase_set::pmap order) and pack their coordinates on the device.
#ifndef ALETSCH_B200_CSRC_K_PHASE_H
#define ALETSCH_B200_CSRC_K_PHASE_H

#include "k_bridge.h"

namespace agpu {

struct phase_dev
{
	const int64_t *frg_off;          // [NB+1]
	const int32_t *f_bundle, *f_h1, *f_h2, *f_type;
	const int32_t *hit_bundle;
	chains_view hc, fc;
	const int32_t *hit_chain;        // hcst handle of every hit (bundle-local chain index, -1)
	const int32_t *frag_chain;       // fcst handle of every fragment, or NULL when no fragment was bridged through a chain
	int32_t *fb;                     // [H] -1 untouched, 0 paired and waiting, 1 covered by a bridged fragment
	int32_t *len;                    // [F+H] coordinates of the element's list, 0 if it contributes none
	int32_t *elem_bundle;            // [F+H]
	const int64_t *off;              // scanned len (pass 1)
	int32_t *val;
};

// the list without its two end coordinates, as up to three pieces
DEV bool phase_middle(const phase_dev &p, int b, int type, int64_t f, int64_t i1, int64_t i2, seq3 &xy)
{
	const int32_t *v1 = NULL, *v2 = NULL;
	int n1 = 0, n2 = 0;
	if(p.hit_chain[i1] >= 0) { v1 = p.hc.ptr(b, p.hit_chain[i1]); n1 = p.hc.len(b, p.hit_chain[i1]); }
	if(i2 >= 0 && p.hit_chain[i2] >= 0) { v2 = p.hc.ptr(b, p.hit_chain[i2]); n2 = p.hc.len(b, p.hit_chain[i2]); }
	xy.n[0] = xy.n[1] = xy.n[2] = 0;
	xy.p[0] = xy.p[1] = xy.p[2] = v1;
	if(type == 1) return merge_intron_chains(v1, n1, v2, n2, xy);
	xy.p[0] = v1; xy.n[0] = n1;
	if(type >= 2)
	{
		int fc = p.frag_chain ? p.frag_chain[f] : -1;
		if(fc >= 0) { xy.p[1] = p.fc.ptr(b, fc); xy.n[1] = p.fc.len(b, fc); }
		xy.p[2] = v2; xy.n[2] = n2;
	}
	return true;
}

DEV bool phase_increasing(int32_t p1, const seq3 &xy, int32_t p2)
{
	int n = xy.size();
	if(n == 0) return p1 <= p2;
	if(p1 > xy.at(0) || xy.at(n - 1) > p2) return false;
	return seq_increasing(xy);
}

// one thread per fragment; emit = 0: decide + measure (and mark the hits), emit = 1: write the coordinates
KERNEL k_phase_frag(int64_t n_frg, int emit, hits_dev h, graph_dev g, phase_dev p)
{
	int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(f >= n_frg) return;
	const int b = p.f_bundle[f];
	const int64_t h0 = h.bundle_hit_off[b];
	const int64_t e = f + h0;                        // E_off[b] + (f - frg_off[b])
	if(!emit) { p.len[e] = 0; p.elem_bundle[e] = b; }
	else if(p.len[e] == 0) return;
	const int t = p.f_type[f];
	if(t <= -1) return;
	const int64_t i1 = h0 + p.f_h1[f], i2 = h0 + p.f_h2[f];
	if(t == 0) { if(!emit) { p.fb[i1] = 0; p.fb[i2] = 0; } return; }
	gview gv = graph_of(g, b);
	int u1 = locate_vertex(gv, h.pos[i1]), u2 = locate_vertex(gv, h.rpos[i2] - 1);
	if(u1 < 0 || u2 < 0) return;
	const int32_t p1 = gv.v_l[u1], p2 = gv.v_r[u2];
	seq3 xy;
	if(!phase_middle(p, b, t, f, i1, i2, xy)) return;
	if(!phase_increasing(p1, xy, p2)) return;
	const int n = xy.size();
	if(!emit) { p.fb[i1] = 1; p.fb[i2] = 1; p.len[e] = n + 2; return; }
	int32_t *out = p.val + p.off[e];
	out[0] = p1;
	for(int k = 0; k < n; k++) out[1 + k] = xy.at(k);
	out[n + 1] = p2;
}

// one thread per hit that no fragment accounted for
KERNEL k_phase_hit(int64_t n_hits, int emit, hits_dev h, graph_dev g, phase_dev p)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_hits) return;
	const int b = p.hit_bundle[i];
	const int64_t e = i + p.frg_off[b + 1];          // E_off[b] + F_b + (i - hit_off[b])
	if(!emit) { p.len[e] = 0; p.elem_bundle[e] = b; }
	else if(p.len[e] == 0) return;
	if(p.fb[i] >= 0) return;
	gview gv = graph_of(g, b);
	int u1 = locate_vertex(gv, h.pos[i]), u2 = locate_vertex(gv, h.rpos[i] - 1);
	if(u1 < 0 || u2 < 0) return;
	const int32_t p1 = gv.v_l[u1], p2 = gv.v_r[u2];
	seq3 xy;
	phase_middle(p, b, 0, -1, i, -1, xy);
	if(!phase_increasing(p1, xy, p2)) return;
	const int n = xy.size();
	if(!emit) { p.len[e] = n + 2; return; }
	int32_t *out = p.val + p.off[e];
	out[0] = p1;
	for(int k = 0; k < n; k++) out[1 + k] = xy.at(k);
	out[n + 1] = p2;
}

// phase_set::add (rnacore/phase_set.cc:12-25): merge equal lists, count them; uniq[e] = 0 for the element that represents
// its list, else -1.  cnt: the count every element adds (NULL: 1 each).  Regions are per bundle, or per cluster when the
// elements are the distinct phases of the cluster's members (phase_set::combine); a combined count is at most the fragments
// plus hits of the cluster's members, far below 2^31 in any batch under the batching rule (include/aletsch_gpu.h), so int32
// holds it.
KERNEL k_phase_insert(int64_t n_elem, const int32_t *elem_bundle, const int32_t *len, const int64_t *off, const int32_t *val,
		const int64_t *reg_off, u64 *slot_word, int32_t *slot_cnt, int64_t *elem_slot, int *err, const int32_t *cnt)
{
	int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(e >= n_elem) return;
	elem_slot[e] = -1;
	if(len[e] <= 0) return;
	const int b = elem_bundle[e];
	chain_src s;
	s.val = val; s.off = off; s.off32 = NULL; s.len = len;
	int64_t r0 = reg_off[b];
	u32 rs = (u32)(reg_off[b + 1] - r0);
	int64_t sl = chain_table_insert(slot_word, r0, rs, s, e, chain_hash(val + off[e], len[e]));
	elem_slot[e] = sl;
	if(sl < 0) { atomicAdd(&err[ERR_CAP], 1); return; }
	atomicAdd(&slot_cnt[sl], cnt ? cnt[e] : 1);
}

KERNEL k_phase_uniq_flag(int64_t n_elem, const int64_t *elem_slot, const u64 *slot_word, int32_t *uniq)
{
	int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(e >= n_elem) return;
	int64_t sl = elem_slot[e];
	uniq[e] = (sl >= 0 && (int64_t)(u32)(slot_word[sl] & 0xffffffffULL) - 1 == e) ? 0 : -1;
}

KERNEL k_phase_compact(int64_t n_elem, const int32_t *uniq, const int64_t *urank, const int64_t *elem_slot, const int32_t *slot_cnt,
		const int64_t *off, const int32_t *len, int64_t *u_off, int32_t *u_len, int32_t *u_cnt)
{
	int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(e >= n_elem || uniq[e] < 0) return;
	int64_t k = urank[e];
	u_off[k] = off[e]; u_len[k] = len[e]; u_cnt[k] = slot_cnt[elem_slot[e]];
}

// E_off[b] = frg_off[b] + hit_off[b]
KERNEL k_phase_elem_off(int64_t n, const int64_t *frg_off, const int64_t *hit_off, int64_t *e_off)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	e_off[i] = frg_off[i] + hit_off[i];
}

// ---- combined phase sets of bundle clusters (assembler::assemble(vector<bundle*>), meta/assembler.cc:177-373: px.combine(ps)
// for every member).  The elements are the distinct phases of every member, cluster by cluster, members in the caller's order.

// distinct phases of member j (bundle members[j])
KERNEL k_gphase_member_count(int64_t n_members, const int32_t *members, const int64_t *boff, int32_t *cnt)
{
	int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(j >= n_members) return;
	const int m = members[j];
	cnt[j] = (int32_t)(boff[m + 1] - boff[m]);
}

// element e of member j = phase boff[members[j]] + (e - moff[j]): its coordinates (offset into the members' ph_val, length),
// count and cluster
KERNEL k_gphase_elements(int64_t n_elem, int32_t n_members, const int64_t *moff, const int32_t *members, const int32_t *member_group,
		const int64_t *boff, const int64_t *ph_off, const int32_t *ph_len, const int32_t *ph_cnt,
		int64_t *e_off, int32_t *e_len, int32_t *e_cnt, int32_t *e_group)
{
	int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(e >= n_elem) return;
	const int j = find_segment(moff, n_members, e);
	const int64_t src = boff[members[j]] + (e - moff[j]);
	e_off[e] = ph_off[src]; e_len[e] = ph_len[src]; e_cnt[e] = ph_cnt[src]; e_group[e] = member_group[j];
}

// ---- phase_set::pmap order (std::map<vector<int32_t>, int>: std::lexicographical_compare on signed int32) of the distinct
// lists of every segment (a bundle, or a cluster).  Lists of segment s are [seg_off[s], seg_off[s + 1]); they are distinct, so
// the order is total.  Every list gets a 64-bit key of its first two coordinates (sign bit flipped; 0 for a missing one), and a
// bitonic network orders (key, index in the segment) pairs, comparing the full lists only where the keys are equal.  A segment
// of at most PHASE_SORT_SMEM_MAX lists is ordered by one CTA in shared memory; larger ones by one launch per network step
// over all their lists, in global memory.
#define PHASE_SORT_SMEM_MAX 2048

struct phase_lists
{
	const int64_t *off;
	const int32_t *len;
	const int32_t *val;
};

// full lexicographic compare of lists x and y (a proper prefix comes first); the index breaks ties between equal lists
DEV bool phase_list_less(const phase_lists &L, int64_t x, int64_t y)
{
	const int32_t *a = L.val + L.off[x], *b = L.val + L.off[y];
	const int na = L.len[x], nb = L.len[y], n = na < nb ? na : nb;
	for(int k = 0; k < n; k++) if(a[k] != b[k]) return a[k] < b[k];
	if(na != nb) return na < nb;
	return x < y;
}

DEV bool phase_order_less(u64 ka, u32 ia, u64 kb, u32 ib, const phase_lists &L, int64_t base)
{
	if(ka != kb) return ka < kb;
	return phase_list_less(L, base + ia, base + ib);
}

// one thread per list: its segment, key and index in the segment
KERNEL k_phase_order_init(int64_t n, int32_t n_seg, const int64_t *seg_off, phase_lists L, int32_t *seg, u64 *key, u32 *idx)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	const int s = find_segment(seg_off, n_seg, i);
	const int32_t *v = L.val + L.off[i];
	const int len = L.len[i];
	const u64 hi = len > 0 ? (u64)((u32)v[0] ^ 0x80000000u) : 0, lo = len > 1 ? (u64)((u32)v[1] ^ 0x80000000u) : 0;
	seg[i] = s; key[i] = hi << 32 | lo; idx[i] = (u32)(i - seg_off[s]);
}

// one CTA per segment of 2 .. bound lists: the network in shared memory; idx[] of the segment is left in order
KERNEL k_phase_order_smem(int32_t n_seg, const int64_t *seg_off, int64_t bound, phase_lists L, const u64 *key, u32 *idx)
{
	SHARED u64 sk[PHASE_SORT_SMEM_MAX];
	SHARED u32 si[PHASE_SORT_SMEM_MAX];
	for(int s = blockIdx.x; s < n_seg; s += gridDim.x)
	{
		const int64_t base = seg_off[s];
		const int n = (int)(seg_off[s + 1] - base);
		if(n < 2 || n > bound) continue;
		for(int i = threadIdx.x; i < n; i += blockDim.x) { sk[i] = key[base + i]; si[i] = idx[base + i]; }
		BLOCK_SYNC();
		for(int k = 2; (k >> 1) < n; k <<= 1)
			for(int j = k >> 1, first = 1; j > 0; j >>= 1, first = 0)
			{
				for(int i = threadIdx.x; i < n; i += blockDim.x)
				{
					int p = first ? (i ^ (k - 1)) : (i ^ j);
					if(p > i && p < n && phase_order_less(sk[p], si[p], sk[i], si[i], L, base))
					{
						u64 tk = sk[i]; sk[i] = sk[p]; sk[p] = tk;
						u32 ti = si[i]; si[i] = si[p]; si[p] = ti;
					}
				}
				BLOCK_SYNC();
			}
		for(int i = threadIdx.x; i < n; i += blockDim.x) idx[base + i] = si[i];
		BLOCK_SYNC();
	}
}

// one step (k, j) of the same network over the segments of more than `bound` lists, in place in global memory; one thread per
// list, the lower index of every pair does the compare-exchange.  Steps past a segment's own network leave it as it is (all
// compare-exchanges are ascending), and are skipped.
KERNEL k_phase_order_step(int64_t n, int64_t k, int64_t j, int first, const int32_t *seg, const int64_t *seg_off, int64_t bound,
		phase_lists L, u64 *key, u32 *idx)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	const int s = seg[i];
	const int64_t base = seg_off[s], ns = seg_off[s + 1] - base;
	if(ns <= bound || (k >> 1) >= ns) return;
	const int64_t li = i - base, p = first ? (li ^ (k - 1)) : (li ^ j);
	if(p <= li || p >= ns) return;
	const int64_t a = base + li, b = base + p;
	if(phase_order_less(key[b], idx[b], key[a], idx[a], L, base))
	{
		u64 tk = key[a]; key[a] = key[b]; key[b] = tk;
		u32 ti = idx[a]; idx[a] = idx[b]; idx[b] = ti;
	}
}

// the view in order: list i of the output is list src[i] = seg_off[seg[i]] + idx[i]; its length and count
KERNEL k_phase_pack_len(int64_t n, const int32_t *seg, const int64_t *seg_off, const u32 *idx, const int32_t *len, const int32_t *cnt,
		int64_t *src, int32_t *olen, int32_t *ocnt)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	const int64_t x = seg_off[seg[i]] + idx[i];
	src[i] = x; olen[i] = len[x]; ocnt[i] = cnt[x];
}

// its coordinates at the scanned offsets (one thread per list: lists are a few coordinates long)
KERNEL k_phase_pack_val(int64_t n, const int64_t *src, phase_lists L, const int64_t *co, int32_t *out)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	const int64_t x = src[i];
	const int32_t *v = L.val + L.off[x];
	int32_t *o = out + co[i];
	for(int k = 0, m = L.len[x]; k < m; k++) o[k] = v[k];
}

} // namespace agpu

#endif
