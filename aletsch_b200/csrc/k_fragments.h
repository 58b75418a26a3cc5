// Stage 3a kernels: mate pairing (bundle_base::build_fragments, rnacore/bundle_base.cc:267-323).
//
// Reference semantics: for i ascending, an unpaired hit i takes the first unpaired u != i (in index
// order) with hits[u].pos == hits[i].mpos, isize sum 0 and the same qname; frgs is ordered by i.
// The bucket hash of the reference only accelerates the search, so the result is a function of the
// candidate relation C(i) = { u != i : pos[u] == mpos[i], isize[u] == -isize[i], qname[u] == qname[i] } alone.
//
// The hits of a bundle arrive sorted by pos (packing contract, verified by k_hit_bounds), so C(i) is a
// run of the bundle's own pos array: a JOIN ON THE SORTED POSITIONS finds it by bisection, and no table of
// query names is built at all (the batch-wide open-addressing table this replaces was 32 bytes per hit
// -- 750 MB at configs[1] -- and crossed the DRAM bus three times).
//   k_pair_probe  : one thread per hit: bisection of the bundle's pos array for mpos -- first over every 64th position
//                   (k_pos_sample: 1/64 of the array, L1-resident for a bundle's slice), then inside the 64 positions
//                   between two samples -- then the walk of the run, recording cand[i] (-1 none, >= 0 the only candidate,
//                   -2 several) and want[u]++ for every candidate u.  (A variant that staged the positions of a tile of
//                   1024 hits and 3584 neighbours on either side in shared memory measured 0.53 ms against 0.46 ms at
//                   configs[1]: the deep bundles, whose mates lie thousands of hits away, fell back to global bisection.)
//   k_pair_decide : the component of the candidate relation a hit lies in is CLOSED and of size two when
//                   C(i) = {u}, nobody but i wants u, C(u) is empty or {i} and nobody but (possibly) u wants i:
//                   the reference's greedy pairs such a component whatever else the bundle holds, discovered by i
//                   (u's candidate list empty) or by the smaller index (mutual).  Every other hit that has or is a
//                   candidate is marked (bit 31 of want[]) together with all its candidates; the marked hits are
//                   exactly the members of the components that are not such pairs.
//                   A bundle in which some mate position holds more than run_max (1024, AGPU_PAIR_RUN_MAX) hits is marked as a
//                   whole, so a hit never walks a longer run: R reads at one start position cost R table operations there,
//                   not R^2 comparisons.
//   k_pairx_*     : the marked hits (multi-mapped query names inside one bundle; none in most batches) go through
//                   the exact greedy per (bundle, qname) group: compact list, open-addressing table sized for the
//                   list, member lists sorted by hit index, pair_group.  Unmarked hits never appear in a marked
//                   hit's candidate list, so running the greedy on the marked members of a group alone is exact.
#ifndef ALETSCH_B200_CSRC_K_FRAGMENTS_H
#define ALETSCH_B200_CSRC_K_FRAGMENTS_H

#include "runtime.h"
#include "k_evidence.h"

namespace agpu {

#define QID_EMPTY 0xffffffffffffffffULL
#define SCAN_TILE 2048

#define PC_NONE (-1)
#define PC_MULTI (-2)
#define WANT_MARK 0x80000000u

// pair control words of a batch: [0] hits marked for the exact path, [1] cursor of the compact list, [2] cursor of the member scratch
enum { PCTL_MARKED = 0, PCTL_LIST, PCTL_MEMBERS, PCTL_WORDS = 4 };

// walks the run of pos == mpos[i] that starts at hit `lo` of i's bundle (which ends at h1) and calls f(u) for every candidate
template<typename F> DEV void pair_candidates(const hits_dev &h, int64_t i, int64_t lo, int64_t h1, F f)
{
	const int32_t m = h.mpos[i];
	const u32 is = (u32)h.isize[i];
	const u64 key = h.qid[i];
	for(int64_t u = lo; u < h1 && h.pos[u] == m; u++)
	{
		if(u == i) continue;
		if((u32)h.isize[u] + is != 0u) continue;
		if(h.qid[u] != key) continue;
		f(u);
	}
}

// pos64[j] = pos[64 j] over the whole batch (1/64 of the positions: the slice of a deep bundle stays in L1); a hit bisects the
// samples that lie inside its bundle, then the 64 positions between two samples
#define PS_STEP 64
KERNEL k_pos_sample(hits_dev h, int64_t n_samples, int32_t *pos64)
{
	const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(j >= n_samples) return;
	pos64[j] = h.pos[j * PS_STEP];
}

// first hit of the bundle [h0, h1) whose pos is >= m
DEV int64_t sampled_lower_bound(const int32_t *pos, const int32_t *pos64, int64_t h0, int64_t h1, int32_t m)
{
	int64_t lo = h0, hi = h1;                                  // the answer lies in [lo, hi]
	const int64_t j0 = (h0 + PS_STEP - 1) / PS_STEP, j1 = (h1 - 1) / PS_STEP;      // samples inside the bundle: j0 .. j1
	if(h1 > h0 && j0 <= j1)
	{
		const int64_t js = j0 + lower_bound_idx(pos64 + j0, (int)(j1 - j0 + 1), m);   // first sample >= m (j1 + 1: none)
		if(js > j0) lo = (js - 1) * PS_STEP + 1;
		if(js <= j1) hi = js * PS_STEP;
	}
	return lo + lower_bound_idx(pos + lo, (int)(hi - lo), m);
}

// run_max: a run of more than run_max hits at the mate position is not walked (a walk per hit that points there would make a
// bundle with R reads at one start position cost R^2, which the reference's bucketed search does not); the hit's whole BUNDLE
// then goes through the exact path, whose table finds a name in O(1) -- components never leave a bundle, so that is closed.
KERNEL k_pair_probe(hits_dev h, const int32_t *pos64, const int32_t *hit_bundle, int32_t *cand, u32 *want, int32_t *bundle_exact, int run_max, int *err)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= h.n_hits) return;
	const u64 key = h.qid[i];
	const int32_t m = h.mpos[i];
	const u32 is = (u32)h.isize[i];
	const int b = hit_bundle[i];
	if(key == QID_EMPTY) { atomicAdd(&err[ERR_QID], 1); cand[i] = PC_NONE; return; }
	const int64_t h0 = h.bundle_hit_off[b], h1 = h.bundle_hit_off[b + 1];
	int n = 0;
	int64_t first = -1;
	const int64_t lo = sampled_lower_bound(h.pos, pos64, h0, h1, m);
	for(int64_t u = lo; u < h1 && h.pos[u] == m; u++)
	{
		// (the want[] counts left behind do not matter: no hit of the bundle takes the direct path)
		if(u - lo >= run_max) { bundle_exact[b] = 1; cand[i] = PC_MULTI; return; }
		const u32 iu = (u32)h.isize[u];
		const u64 ku = h.qid[u];                               // loaded next to isize, not after it
		if(u == i || iu + is != 0u || ku != key) continue;
		if(n == 0) first = u;
		n++;
		atomicAdd(&want[u], 1u);
	}
	cand[i] = n == 0 ? PC_NONE : n == 1 ? (int32_t)(first - h0) : PC_MULTI;
}

DEV void pair_mark(u32 *want, int64_t x, int32_t *ctl)
{
	const u32 old = atomicOr(&want[x], WANT_MARK);
	if(!(old & WANT_MARK)) atomicAdd(&ctl[PCTL_MARKED], 1);
}

// all: every hit that has a candidate goes to the exact path (test hook, AGPU_PAIR_EXACT=1)
KERNEL k_pair_decide(hits_dev h, const int32_t *pos64, const int32_t *hit_bundle, const int32_t *cand, u32 *want, const int32_t *bundle_exact,
		int32_t *mate, int32_t *ctl, int all)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= h.n_hits) return;
	const int32_t c = cand[i];
	const int b = hit_bundle[i];
	if(bundle_exact[b]) { pair_mark(want, i, ctl); return; }      // every hit of such a bundle, candidates or not
	if(c == PC_NONE) return;
	const int64_t h0 = h.bundle_hit_off[b], h1 = h.bundle_hit_off[b + 1];
	const int32_t li = (int32_t)(i - h0);
	if(c >= 0 && !all)
	{
		const int64_t u = h0 + c;
		const u32 wu = want[u] & ~WANT_MARK, wi = want[i] & ~WANT_MARK;
		const int32_t cu = cand[u];
		if(wu == 1 && ((cu == PC_NONE && wi == 0) || (cu == li && wi == 1)))
		{
			if(cu == PC_NONE || li < c) { mate[i] = c; mate[u] = -2 - li; }      // i discovered the pair
			return;
		}
	}
	pair_mark(want, i, ctl);
	const int64_t lo = sampled_lower_bound(h.pos, pos64, h0, h1, h.mpos[i]);
	pair_candidates(h, i, lo, h1, [&](int64_t u) { pair_mark(want, u, ctl); });
}

// the reference's greedy over one qname group whose members m[0..n) are in ascending hit index
DEV void pair_group(const hits_dev &h, int64_t h0, const int32_t *m, int n, int32_t *mate)
{
	for(int a = 0; a < n; a++)
	{
		int64_t ia = h0 + m[a];
		if(mate[ia] != -1) continue;
		for(int c = 0; c < n; c++)
		{
			if(c == a) continue;
			int64_t ic = h0 + m[c];
			if(mate[ic] != -1) continue;
			if(h.pos[ic] != h.mpos[ia]) continue;
			if((u32)h.isize[ic] + (u32)h.isize[ia] != 0u) continue;
			mate[ia] = m[c];                 // i discovered the pair
			mate[ic] = -2 - m[a];            // partner
			break;
		}
	}
}

// ---- exact path over the marked hits
KERNEL k_pairx_list(int64_t n_hits, const u32 *want, int32_t *ctl, int64_t *clist)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_hits) return;
	if(want[i] & WANT_MARK) clist[atomicAdd(&ctl[PCTL_LIST], 1)] = i;
}

// rep[p] = the marked hit that claimed slot p (QID_EMPTY when free); equality is checked on (bundle, key) of the claimant, so
// hash collisions only cost a probe.  head[p] / nextx[t] chain the list positions t of a group.  The table has at least twice
// as many slots as there are marked hits.
KERNEL k_pairx_insert(hits_dev h, int64_t n_c, const int64_t *clist, const int32_t *hit_bundle, u64 mask, u64 *rep, u64 *head, u64 *nextx, u64 *slot_of)
{
	const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(t >= n_c) return;
	const int64_t i = clist[t];
	const int b = hit_bundle[i];
	const u64 key = h.qid[i];
	u64 p = mix64(key ^ mix64((u64)(u32)b)) & mask;
	for(;;)
	{
		const u64 cur = atomicCAS(&rep[p], (u64)QID_EMPTY, (u64)i);
		if(cur == QID_EMPTY) break;
		if(hit_bundle[cur] == b && h.qid[cur] == key) break;
		p = (p + 1) & mask;
	}
	slot_of[t] = p;
	nextx[t] = atomicExch(&head[p], (u64)t);
}

// one thread per group (the list position at the head of the group's chain): members in ascending hit index, then the greedy
#define PAIR_LOCAL 8
KERNEL k_pairx_resolve(hits_dev h, int64_t n_c, const int64_t *clist, const int32_t *hit_bundle, const u64 *head, const u64 *nextx, const u64 *slot_of,
		int32_t *ctl, int32_t *members, int32_t *mate)
{
	const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(t >= n_c) return;
	if(head[slot_of[t]] != (u64)t) return;
	const int64_t h0 = h.bundle_hit_off[hit_bundle[clist[t]]];
	int n = 0;
	for(u64 x = (u64)t; x != QID_EMPTY; x = nextx[x]) n++;
	if(n < 2) return;
	int32_t loc[PAIR_LOCAL];
	int32_t *m = loc;
	if(n > PAIR_LOCAL) m = members + atomicAdd(&ctl[PCTL_MEMBERS], n);
	int k = 0;
	for(u64 x = (u64)t; x != QID_EMPTY; x = nextx[x]) m[k++] = (int32_t)(clist[x] - h0);
	for(int a = 1; a < n; a++)               // ascending hit index (insertion sort; groups are tiny)
	{
		const int32_t v = m[a];
		int c = a - 1;
		while(c >= 0 && m[c] > v) { m[c + 1] = m[c]; c--; }
		m[c + 1] = v;
	}
	pair_group(h, h0, m, n, mate);
}

KERNEL k_frag_emit(hits_dev h, const int32_t *hit_bundle, const int32_t *mate, const int64_t *rank, int32_t *f_h1, int32_t *f_h2, int32_t *f_type,
		int32_t *f_bundle)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= h.n_hits) return;
	if(mate[i] < 0) return;
	int64_t f = rank[i];
	f_bundle[f] = hit_bundle[i];
	f_h1[f] = (int32_t)(i - h.bundle_hit_off[hit_bundle[i]]);
	f_h2[f] = mate[i];
	f_type[f] = 0;
}

KERNEL k_gather_i64(int64_t n, const int64_t *idx, const int64_t *src, int64_t *out)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	out[i] = src[idx[i]];
}

} // namespace agpu

struct fragments_state
{
	bool built = false;
	agpu::dbuf<int32_t> mate;
	agpu::dbuf<int64_t> rank, frg_off;
	agpu::dbuf<int32_t> f_h1, f_h2, f_type, f_bundle, bridged;
	int64_t n_frg = 0;
	std::vector<int64_t> frg_off_host;
};

#endif
