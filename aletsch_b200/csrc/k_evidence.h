// Stage 1-2a kernels: per-hit CIGAR walk (coverage difference array + border bitmap, splice
// extraction, chain hashing), chain-set construction, coverage scan -> segments.
//
// Reference semantics reproduced:
//   bundle_base::add_hit            rnacore/bundle_base.cc:73-104   (bundle bounds, dedupe contract)
//   bundle_base::add_intervals      rnacore/bundle_base.cc:106-158  (only BAM_CMATCH adds coverage)
//   hit::extract_splices            rnacore/hit.cc:77-104
//   chain_set::add(v, h, xs)        rnacore/chain_set.cc:64-123     (insertion order, AI3 counts)
//   chain_set::get_splices          rnacore/chain_set.cc:187-210
//   split_interval_map semantics    rnacore/interval_map.h:31       (every inserted border is kept;
//                                                                    zero-valued stretches are absent)
#ifndef ALETSCH_B200_CSRC_K_EVIDENCE_H
#define ALETSCH_B200_CSRC_K_EVIDENCE_H

#include "dev.h"
#include "blockops.h"
#include "lookback.h"

namespace agpu {

#define SCAN1_MAX 1024           // threads of the single-CTA scans
#define COV_ALIGN 128            // bundle windows of the border bitmap start at multiples of 128 positions (4 words)
#define CTILE 2048               // elements per tile of the device-wide scans over border words / borders
#define EMPTY_SLOT 0ULL
#define INT_BIG 0x7fffffff

struct hits_dev
{
	int64_t n_hits;
	int32_t n_bundles;
	const int64_t *bundle_hit_off;
	const int32_t *pos, *rpos, *mpos, *isize;
	const uint16_t *flag;
	const uint8_t *strand, *xs;      // strand may be NULL: then bundle_strand[b] holds the strand all hits of bundle b share
	const uint8_t *bundle_strand;
	const u64 *qid;
	const u32 *cigar_off;
	const u32 *cigar;
};

// error / statistics words shared by all kernels of a batch
enum { ERR_ORDER = 0, ERR_DUP, ERR_STRAND, ERR_RPOS, ERR_LINK, ERR_QID, ERR_CAP, ERR_PACKED, ERR_WORDS = 16 };

// ---- E0: bundle bounds (bundle_base::add_hit) + packing-contract check.  One thread per HIT (bundles range from one hit to
// several hundred thousand: a CTA per bundle leaves the step waiting for the deepest one).  A hit finds its bundle by bisection of
// the offsets -- but a full bisection per hit is a chain of 15 dependent loads that each go to L2 (ncu: 55 % of the stall samples
// of the kernel, 0.35 ms), so k_tile_bundle first bisects once per tile of HB_TILE hits and a hit only searches between the
// bundles of its tile's first hit and of the next tile's (usually the same one: no load at all).  A warp whose hits all lie in
// one bundle reduces first and issues one set of atomics.  k_bundle_init before, k_bundle_finish after (one thread per bundle).
#define HB_TILE 256
// the last bundle whose first hit is not after i (empty bundles in front of it are skipped: their offset equals its own)
DEV int bundle_of_hit(const int64_t *off, int lo, int hi, int64_t i)
{
	while(hi - lo > 1)
	{
		int mid = (lo + hi) >> 1;
		if(off[mid] <= i) lo = mid; else hi = mid;
	}
	return lo;
}
KERNEL k_tile_bundle(hits_dev h, int64_t n_tiles, int32_t *tile_bundle)
{
	const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(t > n_tiles) return;
	const int64_t i = t * HB_TILE;
	tile_bundle[t] = i < h.n_hits ? bundle_of_hit(h.bundle_hit_off, 0, h.n_bundles, i) : h.n_bundles - 1;
}

KERNEL k_bundle_init(int32_t n_bundles, int32_t *b_lpos, int32_t *b_rpos, int32_t *b_covhi, int32_t *b_npq)
{
	int b = blockIdx.x * blockDim.x + threadIdx.x;
	if(b >= n_bundles) return;
	b_lpos[b] = 1 << 30; b_rpos[b] = 0; b_covhi[b] = 0;        // rnacore/bundle_base.cc:21-22
	b_npq[2 * b] = 0; b_npq[2 * b + 1] = 0;
}

KERNEL k_hit_bounds(hits_dev h, const int32_t *tile_bundle, int32_t *b_lpos, int32_t *b_rpos, int32_t *b_covhi, int32_t *b_npq, int32_t *hit_bundle, int *err)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const bool in = i < h.n_hits;
	int b = 0, p = 1 << 30, q = 0, r = 0, np = 0, nq = 0;
	if(in)
	{
		const int64_t t = i / HB_TILE;
		const int blo = tile_bundle[t], bhi = tile_bundle[t + 1];
		b = blo == bhi ? blo : bundle_of_hit(h.bundle_hit_off, blo, bhi + 1, i);
		const int64_t h0 = h.bundle_hit_off[b];
		p = h.pos[i]; r = h.rpos[i];
		const int m = h.mpos[i];
		hit_bundle[i] = b;
		q = r;
		if(m > r && m <= r + 500000) q = m;                    // rnacore/bundle_base.cc:92
		const uint8_t x = h.xs[i];
		np = x == '+'; nq = x == '-';
		if(i > h0)
		{
			if(h.pos[i - 1] > p) atomicAdd(&err[ERR_ORDER], 1);
			if(h.pos[i - 1] == p && h.rpos[i - 1] == r) atomicAdd(&err[ERR_DUP], 1);
			if(h.strand && h.strand[i] != h.strand[i - 1]) atomicAdd(&err[ERR_STRAND], 1);      // (a bundle of one strand has no such neighbours)
		}
	}
#ifndef AGPU_EMU
	const unsigned FULL = 0xffffffffu;
	const int b0 = __shfl_sync(FULL, b, 0);
	if(__all_sync(FULL, in && b == b0))
	{
		p = __reduce_min_sync(FULL, p); q = __reduce_max_sync(FULL, q); r = __reduce_max_sync(FULL, r);
		np = __reduce_add_sync(FULL, np); nq = __reduce_add_sync(FULL, nq);
		if((threadIdx.x & 31) != 0) return;
	}
#endif
	if(!in) return;
	atomicMin(&b_lpos[b], p); atomicMax(&b_rpos[b], q); atomicMax(&b_covhi[b], r);
	if(np) atomicAdd(&b_npq[2 * b], np);
	if(nq) atomicAdd(&b_npq[2 * b + 1], nq);
}

KERNEL k_bundle_finish(hits_dev h, int library_type, const int32_t *b_lpos, const int32_t *b_covhi, const int32_t *b_npq, uint8_t *b_strand, int64_t *b_span)
{
	int b = blockIdx.x * blockDim.x + threadIdx.x;
	if(b >= h.n_bundles) return;
	const int64_t h0 = h.bundle_hit_off[b], h1 = h.bundle_hit_off[b + 1];
	uint8_t st = '.';
	if(h1 > h0) st = h.strand ? h.strand[h0] : h.bundle_strand[b];      // rnacore/bundle_base.cc:100
	if(library_type == 0)                          // bundle_base::compute_strand, rnacore/bundle_base.cc:205-225
	{
		const int np = b_npq[2 * b], nq = b_npq[2 * b + 1];
		if(np > nq) st = '+';
		else if(np < nq) st = '-';
		else st = '.';
	}
	b_strand[b] = st;
	// positions [lpos, covhi] inclusive (the -1 of a block ending at covhi lands there), tile-aligned
	int64_t span = (h1 > h0) ? ((int64_t)b_covhi[b] - (int64_t)b_lpos[b] + 1) : 0;
	b_span[b] = (span + COV_ALIGN - 1) / COV_ALIGN * COV_ALIGN;
}

// ---- device-wide exclusive scan of int64: tile sums, single-CTA scan of the sums, per-tile apply
#define SCAN64_TILE 2048
// hash of one intron chain (length + coordinates)
HD u64 chain_hash(const int32_t *v, int n)
{
	u64 hsh = mix64((u64)n);
	for(int k = 0; k < n; k++) hsh = mix64(hsh ^ (u64)(u32)v[k]);
	return hsh;
}

// ---- E2: one thread per hit: CIGAR walk
//   coverage: a border bit at the start and at the end of every BAM_CMATCH block (the +1 / -1 are added by
//             k_cov_add once the borders have been ranked, see the coverage section below)
//   splices : (p - len, p) for every inner BAM_CREF_SKIP, written at spl[cigar_off[i] ...]
//   skip    : optional per-hit mask (insert-size preview, agpu_batch_coverage_edit): bit z set = the hit's z-th BAM_CMATCH
//             operation adds no coverage
// Every per-hit walk below is a chain of dependent loads (hit -> bundle -> window base, hit -> CIGAR offset -> operation ->
// bitmap word): one hit per thread leaves a thread with one 4-byte load in flight (ncu: 71-77 % of the stall samples on the long
// scoreboard at full occupancy).  A thread therefore takes HQ hits, blockDim.x apart, and issues the loads of each level for all
// of them before it uses any; the first CIGAR operation of a hit (the only one of an unspliced read) is fetched with that level.
// Launch with HQ_THREADS(n_hits) threads.
#define HQ 4
#define HQ_THREADS(n) ((((int64_t)(n) + 256 * HQ - 1) / (256 * HQ)) * 256)
DEV void border_set(u32 *border, int64_t g) { atomicOr(&border[g >> 5], 1u << (g & 31)); }
// (looking at the word first -- a border is asked for 2 times at configs[1], 28 times at configs[4] -- measured slower: the
// load it adds sits in front of the atomic, which otherwise leaves the thread without waiting)
KERNEL k_hit_cigar(hits_dev h, const int32_t *b_lpos, const int64_t *cov_base, u32 *border,
		int32_t *spl, int32_t *hit_nspl, const int32_t *hit_bundle, int32_t *n_spliced, int *err, const uint16_t *skip)
{
	const int64_t i0 = (int64_t)blockIdx.x * blockDim.x * HQ + threadIdx.x;
	int bq[HQ];
	u32 c0q[HQ], c1q[HQ], skq[HQ], firstq[HQ];
	int32_t pq[HQ], rq[HQ];
	int64_t baseq[HQ];
#pragma unroll
	for(int q = 0; q < HQ; q++)
	{
		const int64_t i = i0 + (int64_t)q * blockDim.x;
		const bool in = i < h.n_hits;
		bq[q] = in ? hit_bundle[i] : -1;
		c0q[q] = in ? h.cigar_off[i] : 0u;
		c1q[q] = in ? h.cigar_off[i + 1] : 0u;
		pq[q] = in ? h.pos[i] : 0;
		rq[q] = in ? h.rpos[i] : 0;
		skq[q] = (in && skip) ? skip[i] : 0u;
	}
#pragma unroll
	for(int q = 0; q < HQ; q++)
	{
		baseq[q] = bq[q] >= 0 ? cov_base[bq[q]] - (int64_t)b_lpos[bq[q]] : 0;
		firstq[q] = c1q[q] > c0q[q] ? h.cigar[c0q[q]] : 0u;
	}
#pragma unroll
	for(int q = 0; q < HQ; q++)
	{
		const int b = bq[q];
		if(b < 0) continue;
		const int64_t i = i0 + (int64_t)q * blockDim.x;
		const int64_t base = baseq[q];
		const u32 c0 = c0q[q], c1 = c1q[q], sk = skq[q];
		int32_t p = pq[q];
		int ns = 0, z = 0;
		int32_t *out = spl + c0;
		for(u32 k = c0; k < c1; k++)
		{
			const u32 c = k == c0 ? firstq[q] : h.cigar[k];
			const u32 op = c & 0xf, len = c >> 4;
			if((0x3C1A7 >> (op << 1)) & 2) p += (int32_t)len;      // bam_cigar_type: consumes reference
			if(op == 0)                                            // BAM_CMATCH
			{
				const int64_t s = base + p - (int32_t)len, e = base + p;
				const bool skipped = z < 16 && ((sk >> z) & 1u);
				z++;
				if(len > 0 && !skipped) { border_set(border, s); border_set(border, e); }
			}
			if(op == 3 && k != c0 && k != c1 - 1)                  // BAM_CREF_SKIP, not first / last op
			{
				out[ns++] = p - (int32_t)len;
				out[ns++] = p;
			}
		}
		if(p != rq[q]) atomicAdd(&err[ERR_RPOS], 1);
		hit_nspl[i] = ns;
#ifndef AGPU_EMU
		// hits of a bundle are neighbours: one atomic per (warp, bundle) instead of one per spliced hit
		const unsigned act = __activemask();
		const unsigned peers = __match_any_sync(act, ns > 0 ? b : -1);
		if(ns > 0 && (int)(threadIdx.x & 31) == __ffs((int)peers) - 1) atomicAdd(&n_spliced[b], __popc(peers));
#else
		if(ns > 0) atomicAdd(&n_spliced[b], 1);
#endif
	}
}

// hit.rpos = pos + bam_cigar2rlen (rnacore/hit.cc:64) when the host did not send it
KERNEL k_hit_rpos(hits_dev h, int32_t *rpos)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= h.n_hits) return;
	u32 c0 = h.cigar_off[i], c1 = h.cigar_off[i + 1];
	int32_t p = h.pos[i];
	for(u32 k = c0; k < c1; k++)
	{
		u32 c = h.cigar[k];
		if((0x3C1A7 >> ((c & 0xf) << 1)) & 2) p += (int32_t)(c >> 4);
	}
	rpos[i] = p;
}

// chain table region of a bundle: a power of two >= 2 x the elements that carry a chain
KERNEL k_table_sizes(int64_t nb, const int32_t *count, int64_t *size)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= nb) return;
	int c = 2 * count[i];
	size[i] = (int64_t)pow2_ceil((u32)(c < 2 ? 2 : c));
}

// the same from an offset array: count = off[i + 1] - off[i]
KERNEL k_table_sizes_off(int64_t nb, const int64_t *off, int64_t *size)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= nb) return;
	int64_t c = 2 * (off[i + 1] - off[i]);
	size[i] = (int64_t)pow2_ceil((u32)(c < 2 ? 2 : c));
}

KERNEL k_add_i64(int64_t n, const int64_t *a, const int64_t *b, int64_t *out)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	out[i] = a[i] + b[i];
}

// ---- chain table: one open-addressing region per bundle; slot word = hash32 << 32 | (rep + 1)
// `rep` is the global index of the element that claimed the slot; equality is verified on the
// actual coordinates, so hash collisions only cost a probe.
struct chain_src
{
	const int32_t *val;        // coordinates
	const int64_t *off;        // element e owns val[off[e] .. off[e] + len[e])   (NULL: use off32)
	const u32 *off32;
	const int32_t *len;
	HD const int32_t *ptr(int64_t e) const { return val + (off ? off[e] : (int64_t)off32[e]); }
};

HD bool same_chain(const chain_src &s, int64_t a, int64_t b)
{
	int n = s.len[a];
	if(n != s.len[b]) return false;
	const int32_t *x = s.ptr(a), *y = s.ptr(b);
	for(int k = 0; k < n; k++) if(x[k] != y[k]) return false;
	return true;
}

// returns the slot (global index) holding the chain of element e, inserting it if new
DEV int64_t chain_table_insert(u64 *slot_word, int64_t reg0, u32 reg_size, const chain_src &s, int64_t e, u64 hsh)
{
	u32 mask = reg_size - 1;
	u32 pos = (u32)(hsh >> 7) & mask;
	u64 mine = ((hsh >> 32) << 32) | (u64)(u32)(e + 1);
	for(u32 probe = 0; probe <= mask; probe++)
	{
		u64 cur = atomicCAS(&slot_word[reg0 + pos], (u64)EMPTY_SLOT, mine);
		if(cur == EMPTY_SLOT) return reg0 + pos;
		if((cur >> 32) == (mine >> 32))
		{
			int64_t rep = (int64_t)(u32)(cur & 0xffffffffULL) - 1;
			if(same_chain(s, rep, e)) return reg0 + pos;
		}
		pos = (pos + 1) & mask;
	}
	return -1;
}

// ---- E3: one thread per hit with splices: insert into hcst table, count xs class, track first hit
KERNEL k_hcst_insert(hits_dev h, const int32_t *hit_nspl, const int32_t *hit_bundle, const int32_t *spl,
		const int64_t *reg_off, u64 *slot_word, int32_t *slot_first, int32_t *slot_cnt, int64_t *hit_slot, int *err)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= h.n_hits) return;
	hit_slot[i] = -1;
	if(hit_nspl[i] <= 0) return;
	int b = hit_bundle[i];
	chain_src s;
	s.val = spl; s.off = NULL; s.off32 = h.cigar_off; s.len = hit_nspl;
	int64_t r0 = reg_off[b];
	u32 rs = (u32)(reg_off[b + 1] - r0);
	int64_t sl = chain_table_insert(slot_word, r0, rs, s, i, chain_hash(spl + h.cigar_off[i], hit_nspl[i]));
	if(sl < 0) { atomicAdd(&err[ERR_CAP], 1); return; }
	hit_slot[i] = sl;
	int x = 0;
	if(h.xs[i] == '+') x = 1;
	if(h.xs[i] == '-') x = 2;
	atomicAdd(&slot_cnt[sl * 3 + x], 1);
	atomicMin(&slot_first[sl], (int32_t)(i - h.bundle_hit_off[b]));
}

// ---- E4: per bundle: order the chains the way chain_set::add leaves them
// (groups by first appearance of the first coordinate, chains by first appearance), number
// them, and build the sorted unique splice list.
KERNEL k_chain_order(const int32_t *order, int32_t n_bundles, const int64_t *elem_off, const int64_t *hit_slot, const int32_t *slot_first,
		const int32_t *slot_cnt, const u32 *elem_voff32, const int64_t *elem_voff64, const int32_t *val,
		u64 *key_scratch, int32_t *slot_chain,
		int32_t *n_chains, int32_t *c_rep, int32_t *c_cnt, int32_t *c_grp, int64_t *c_slot)
{
	SHARED int s_n;
	for(int bi = blockIdx.x; bi < n_bundles; bi += gridDim.x)
	{
		const int b = order ? order[bi] : bi;
		int64_t e0 = elem_off[b], e1 = elem_off[b + 1];
		int ne = (int)(e1 - e0);
		u64 *key = key_scratch + e0;
		int32_t *tmp = c_grp + e0;
		if(threadIdx.x == 0) s_n = 0;
		BLOCK_SYNC();
		// chain heads: elements that are the first appearance of their chain
		for(int i = threadIdx.x; i < ne; i += blockDim.x)
		{
			int64_t sl = hit_slot[e0 + i];
			if(sl >= 0 && slot_first[sl] == i)
			{
				int k = atomicAdd(&s_n, 1);
				const int32_t *v = val + (elem_voff64 ? elem_voff64[e0 + i] : (int64_t)elem_voff32[e0 + i]);
				key[k] = ((u64)(u32)v[0] << 32) | (u64)(u32)i;        // (first coordinate, first element)
			}
		}
		BLOCK_SYNC();
		int nc = s_n;
		block_sort_u64(key, nc);
		// a group's rank is the first element that opened it = low word of the group's first key
		for(int k = threadIdx.x; k < nc; k += blockDim.x)
			tmp[k] = (k == 0 || (key[k - 1] >> 32) != (key[k] >> 32)) ? k : 0;
		BLOCK_SYNC();
		block_incl_maxscan(tmp, nc);
		for(int k = threadIdx.x; k < nc; k += blockDim.x)
			c_rep[e0 + k] = (int32_t)(u32)(key[tmp[k]] & 0xffffffffULL);
		BLOCK_SYNC();
		for(int k = threadIdx.x; k < nc; k += blockDim.x)
			key[k] = ((u64)(u32)c_rep[e0 + k] << 32) | (key[k] & 0xffffffffULL);   // (group first element, chain first element)
		BLOCK_SYNC();
		block_sort_u64(key, nc);
		// dense group index = number of group changes up to and including k
		for(int k = threadIdx.x; k < nc; k += blockDim.x)
			tmp[k] = (k > 0 && (key[k - 1] >> 32) != (key[k] >> 32)) ? 1 : 0;
		BLOCK_SYNC();
		block_excl_scan(tmp, nc);
		for(int k = threadIdx.x; k < nc; k += blockDim.x)
		{
			int rep = (int)(u32)(key[k] & 0xffffffffULL);
			int64_t sl = hit_slot[e0 + rep];
			int chg = (k > 0 && (key[k - 1] >> 32) != (key[k] >> 32)) ? 1 : 0;
			c_rep[e0 + k] = rep;
			c_slot[e0 + k] = sl;
			c_cnt[(e0 + k) * 3 + 0] = slot_cnt[sl * 3 + 0];
			c_cnt[(e0 + k) * 3 + 1] = slot_cnt[sl * 3 + 1];
			c_cnt[(e0 + k) * 3 + 2] = slot_cnt[sl * 3 + 2];
			slot_chain[sl] = k;
			tmp[k] = tmp[k] + chg;
		}
		if(threadIdx.x == 0) n_chains[b] = nc;
		BLOCK_SYNC();
	}
}

// per bundle: sorted unique coordinates over all chains with a positive count (chain_set::get_splices)
// scratch regions start at 2 * val_base[b]: n keys followed by n flags
KERNEL k_chain_splices(const int32_t *order, int32_t n_bundles, const int64_t *elem_off, const int64_t *val_base,
		const int32_t *n_chains, const int32_t *c_rep, const int32_t *c_cnt,
		const int32_t *elem_len, const u32 *elem_voff32, const int64_t *elem_voff64, const int32_t *val,
		u64 *key_scratch, int32_t *n_splices, int32_t *splices_scratch)
{
	SHARED int s_n;
	for(int bi = blockIdx.x; bi < n_bundles; bi += gridDim.x)
	{
		const int b = order ? order[bi] : bi;
		int64_t e0 = elem_off[b];
		int nc = n_chains[b];
		u64 *key = key_scratch + 2 * val_base[b];
		if(threadIdx.x == 0) s_n = 0;
		BLOCK_SYNC();
		for(int k = threadIdx.x; k < nc; k += blockDim.x)
		{
			int64_t e = e0 + c_rep[e0 + k];
			if(c_cnt[(e0 + k) * 3] + c_cnt[(e0 + k) * 3 + 1] + c_cnt[(e0 + k) * 3 + 2] <= 0) continue;
			const int32_t *v = val + (elem_voff64 ? elem_voff64[e] : (int64_t)elem_voff32[e]);
			int n = elem_len[e];
			int at = atomicAdd(&s_n, n);
			for(int j = 0; j < n; j++) key[at + j] = (u64)(u32)v[j];
		}
		BLOCK_SYNC();
		int n = s_n;
		block_sort_u64(key, n);
		int *flag = (int*)(key + n);
		for(int i = threadIdx.x; i < n; i += blockDim.x) flag[i] = (i == 0 || key[i] != key[i - 1]) ? 1 : 0;
		BLOCK_SYNC();
		int tot = block_excl_scan(flag, n);
		int32_t *out = splices_scratch + val_base[b];
		for(int i = threadIdx.x; i < n; i += blockDim.x)
			if(i == 0 || key[i] != key[i - 1]) out[flag[i]] = (int32_t)(u32)key[i];
		if(threadIdx.x == 0) n_splices[b] = tot;
		BLOCK_SYNC();
	}
}

// splice lists of all bundles back to back
KERNEL k_splices_compact(int32_t n_bundles, const int64_t *val_base, const int32_t *n_splices, const int32_t *scratch, const int64_t *out_off,
		int32_t *out)
{
	for(int b = blockIdx.x; b < n_bundles; b += gridDim.x)
		for(int i = threadIdx.x; i < n_splices[b]; i += blockDim.x) out[out_off[b] + i] = scratch[val_base[b] + i];
}

// per element: handle -> bundle-local chain index
KERNEL k_handle_chain(int64_t n, const int64_t *hit_slot, const int32_t *slot_chain, int32_t *handle_chain)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	int64_t sl = hit_slot[i];
	handle_chain[i] = sl >= 0 ? slot_chain[sl] : -1;
}

KERNEL k_gather_off(int64_t n, const int64_t *idx, const u32 *src, int64_t *out)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	out[i] = (int64_t)src[idx[i]];
}

// ---- coverage map (bundle_base::mmap, a Boost.ICL split_interval_map) on BORDER-COMPACTED coordinates
//
// split_interval_map semantics (rnacore/interval_map.h:31): every inserted interval end stays a segment border for
// ever, and stretches whose summed value is 0 are absent.  So the map is fully described by (1) the set of borders and
// (2) a +1/-1 difference per border.  Exonic coverage touches only a few percent of a bundle's genomic window, hence:
//   border[L/32]   per-base bitmap of the borders of all bundles' windows (the only per-base structure)
//   wrank[L/32+1]  exclusive prefix popcount of the bitmap words: rank of a position among the borders
//   diffc[NB]      difference array indexed by border rank;   posc[NB] genomic coordinate of every border
// A bundle's differences sum to 0, so ONE device-wide prefix sum over diffc yields every bundle's coverage, and one
// device-wide rank of (coverage > 0) compacts the segments: seg i = (posc[i], posc[i + 1], coverage right of border i).
// Launches (coverage_scan): k_lb_bord_rank (wrank) -- border count read back, it sizes the per-border arrays -- k_bord_off,
// k_bord_positions (posc), the k_cov_add* kernels (diffc), k_lb_cov_segments (coverage, segments, seg_psum, seg_off, run
// heads; the coverage itself is not stored), k_seg_nhead (run structure).  The segment count stays on the device.

// rank of global window position g among the borders (g itself must be a border)
DEV int64_t border_rank(const u32 *border, const u32 *wrank, int64_t g)
{
	u32 w = border[g >> 5];
	return (int64_t)wrank[g >> 5] + __popc(w & ((1u << (g & 31)) - 1u));
}

// one thread per hit: +1 at the start and -1 at the end of every BAM_CMATCH block (bundle_base::add_intervals,
// rnacore/bundle_base.cc:106-158: only op M adds coverage)
KERNEL k_cov_add(hits_dev h, const int32_t *hit_bundle, const int32_t *b_lpos, const int64_t *cov_base, const u32 *border,
		const u32 *wrank, int32_t *diffc, const uint16_t *skip)
{
	const int64_t i0 = (int64_t)blockIdx.x * blockDim.x * HQ + threadIdx.x;       // HQ hits per thread, see k_hit_cigar
	int bq[HQ];
	u32 c0q[HQ], c1q[HQ], skq[HQ], firstq[HQ];
	int32_t pq[HQ];
	int64_t baseq[HQ];
#pragma unroll
	for(int q = 0; q < HQ; q++)
	{
		const int64_t i = i0 + (int64_t)q * blockDim.x;
		const bool in = i < h.n_hits;
		bq[q] = in ? hit_bundle[i] : -1;
		c0q[q] = in ? h.cigar_off[i] : 0u;
		c1q[q] = in ? h.cigar_off[i + 1] : 0u;
		pq[q] = in ? h.pos[i] : 0;
		skq[q] = (in && skip) ? skip[i] : 0u;
	}
#pragma unroll
	for(int q = 0; q < HQ; q++)
	{
		baseq[q] = bq[q] >= 0 ? cov_base[bq[q]] - (int64_t)b_lpos[bq[q]] : 0;
		firstq[q] = c1q[q] > c0q[q] ? h.cigar[c0q[q]] : 0u;
	}
#pragma unroll
	for(int q = 0; q < HQ; q++)
	{
		if(bq[q] < 0) continue;
		const int64_t base = baseq[q];
		const u32 c0 = c0q[q], c1 = c1q[q], sk = skq[q];
		int32_t p = pq[q];
		int z = 0;
		for(u32 k = c0; k < c1; k++)
		{
			const u32 c = k == c0 ? firstq[q] : h.cigar[k];
			const u32 op = c & 0xf, len = c >> 4;
			if((0x3C1A7 >> (op << 1)) & 2) p += (int32_t)len;
			const bool skipped = op == 0 && z < 16 && ((sk >> z) & 1u);
			if(op == 0) z++;
			if(op == 0 && len > 0 && !skipped)
			{
				const int64_t gs = base + p - (int32_t)len, ge = base + p;
				const u32 ws = border[gs >> 5], we = border[ge >> 5];
				const u32 rs = wrank[gs >> 5], re = wrank[ge >> 5];
				atomicAdd(&diffc[(int64_t)rs + __popc(ws & ((1u << (gs & 31)) - 1u))], 1);
				atomicAdd(&diffc[(int64_t)re + __popc(we & ((1u << (ge & 31)) - 1u))], -1);
			}
		}
	}
}

// the stretches added by update_bridges (rnacore/bundle_base.cc:498-504), kept as a list of global window positions
KERNEL k_cov_add_extra(int64_t n, const int64_t *ex_s, const int64_t *ex_e, const u32 *border, const u32 *wrank, int32_t *diffc)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	atomicAdd(&diffc[border_rank(border, wrank, ex_s[i])], 1);
	atomicAdd(&diffc[border_rank(border, wrank, ex_e[i])], -1);
}

// ---- single-pass versions (decoupled look-back, lookback.h) of the coverage scans ------------------------------------------

// wrank[w] = number of borders before bitmap word w (wrank[n_words] = total); *total gets the number of borders
KERNEL k_lb_bord_rank(lb_ctl c, const u32 *border, int64_t n_words, u32 *wrank, int64_t *total)
{
	SHARED16 int f[LB_TILE];
	const int64_t n_tiles = (n_words + 1 + LB_TILE - 1) / LB_TILE;
	for(int64_t t = lb_next_tile(c, n_tiles); t >= 0; t = lb_next_tile(c, n_tiles))
	{
		const int64_t g0 = t * LB_TILE;
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x)
		{
			const int64_t w = g0 + i;
			f[i] = w < n_words ? __popc(border[w]) : 0;
		}
		BLOCK_SYNC();
		const int tot = block_excl_scan(f, LB_TILE);
		const int64_t pre = lb_tile_prefix(c, 0, t, tot);
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x)
		{
			const int64_t w = g0 + i;
			if(w <= n_words) wrank[w] = (u32)(pre + f[i]);
			if(w == n_words) *total = pre + f[i];
		}
	}
}

// bord_off[b] = rank of the first border of bundle b's window (bord_off[NB] = total); tile_b0[k] = first bundle whose first border
// has rank >= k * LB_TILE, for the tiles of k_lb_cov_segments (a bisection of bord_off per tile there sat on every tile's path)
KERNEL k_bord_off(int32_t nb, const int64_t *cov_base, const u32 *wrank, int64_t *bord_off, int64_t n_tiles, int32_t *tile_b0)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i > nb) return;
	const int64_t cur = (int64_t)wrank[cov_base[i] >> 5], prev = i > 0 ? (int64_t)wrank[cov_base[i - 1] >> 5] : -1;
	bord_off[i] = cur;
	for(int64_t k = (prev + LB_TILE) / LB_TILE; k <= cur / LB_TILE && k < n_tiles; k++) tile_b0[k] = (int32_t)i;
}

// genomic coordinate of every border: posc[rank] (posc is sized by the border count, so this runs after it is read back).
// Tiles of LB_TILE words; bundle windows start at multiples of COV_ALIGN positions, so each group of COV_ALIGN / 32 words belongs
// to one bundle: two bisections per tile find the tile's bundles, and every group looks its bundle up among those.
#define BP_GROUP (COV_ALIGN / 32)
KERNEL k_bord_positions(int64_t n_words, const u32 *border, const u32 *wrank, int32_t n_bundles, const int64_t *cov_base,
		const int32_t *b_lpos, int32_t *posc)
{
	SHARED long long s_delta[LB_TILE / BP_GROUP];      // per group of words: b_lpos - cov_base of its bundle
	SHARED int s_b[2];
	const int64_t n_tiles = (n_words + LB_TILE - 1) / LB_TILE;
	for(int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x)
	{
		const int64_t g0 = t * LB_TILE;
		if(threadIdx.x == 0)
		{
			const int64_t last = (g0 + LB_TILE < n_words ? g0 + LB_TILE : n_words) - 1;
			s_b[0] = find_segment(cov_base, n_bundles, g0 << 5);
			s_b[1] = find_segment(cov_base, n_bundles, last << 5);
		}
		BLOCK_SYNC();
		const int b0 = s_b[0], b1 = s_b[1];
		for(int k = threadIdx.x; k < LB_TILE / BP_GROUP; k += blockDim.x)
		{
			const int b = b0 + find_segment(cov_base + b0, b1 - b0, (g0 + (int64_t)k * BP_GROUP) << 5);
			s_delta[k] = b < n_bundles ? (long long)b_lpos[b] - cov_base[b] : 0;
		}
		BLOCK_SYNC();
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x)
		{
			const int64_t w = g0 + i;
			u32 x = w < n_words ? border[w] : 0u;
			if(!x) continue;
			const int32_t p0 = (int32_t)((w << 5) + s_delta[i / BP_GROUP]);
			int64_t o = wrank[w];
			while(x)
			{
				const int k = __ffs((int)x) - 1;
				x &= x - 1;
				posc[o++] = p0 + k;
			}
		}
		BLOCK_SYNC();
	}
}

// differences -> coverage -> segments, one launch.  Three chained look-backs per tile of borders:
//   chain 0: sum of the differences        -> coverage right of every border
//   chain 1: number of borders with coverage > 0 -> position of every segment in the compact list
//   chain 2: sum of the products (r - l) * c of the tile's segments, int32 wrap-around arithmetic -> seg_psum
// Outputs: the segments in order -- border i with coverage c > 0 opens [posc[i], posc[i + 1]) with value c -- as seg_l / seg_r /
// seg_c; seg_head[o] = 1 if segment o does not touch its predecessor (it opens a run of region::build_join_interval_map), else 0;
// seg_psum[o] = the int64 sum of the int32-wrapped product totals of the tiles before o's tile, plus the int32-wrapped sum of the
// products of the segments before o in its tile (seg_psum[n_seg] = total; only differences of nearby entries are read, cut to
// int32: the summands of compute_sum_overlap); seg_off[b] = number of segments before the first border of bundle b; *n_seg.
// Capped at 40 registers for six CTAs per SM: a tile spends most of its time waiting on look-backs, and resident tiles hide that.
KERNEL_OCC(6) k_lb_cov_segments(lb_ctl c, const int32_t *diffc, const int32_t *posc, int64_t n, int32_t n_bundles, const int64_t *bord_off,
		const int32_t *tile_b0, int32_t *seg_l, int32_t *seg_r, int32_t *seg_c, int64_t *seg_off, uint8_t *seg_head, int64_t *seg_psum, int64_t *n_seg)
{
	SHARED16 int f[LB_TILE + 1];     // local prefix of the differences, then of the segment flags
	SHARED int cv[LB_TILE + 1];      // coverage of the tile's borders; cv[LB_TILE]: coverage of the border before the tile
	SHARED16 int pr[LB_TILE];         // products, then their local prefix
	const int64_t n_tiles = (n + 1 + LB_TILE - 1) / LB_TILE;
	for(int64_t t = lb_next_tile(c, n_tiles); t >= 0; t = lb_next_tile(c, n_tiles))
	{
		const int64_t g0 = t * LB_TILE;
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x)
		{
			const int64_t g = g0 + i;
			f[i] = g < n ? diffc[g] : 0;
		}
		BLOCK_SYNC();
		const int dsum = block_excl_scan(f, LB_TILE);
		const int pre = (int)lb_tile_prefix(c, 0, t, dsum);
		// coverage; flags of the segments
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x)
		{
			const int64_t g = g0 + i;
			cv[i] = g < n ? pre + f[i] + diffc[g] : 0;
		}
		if(threadIdx.x == 0) cv[LB_TILE] = pre;      // coverage right of border g0 - 1 = sum of all differences before the tile
		BLOCK_SYNC();
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x)
		{
			const int64_t g = g0 + i;
			const int on = (g < n && cv[i] > 0) ? 1 : 0;
			f[i] = on;
			int32_t p = 0;
			if(on)
			{
				const int32_t pl = posc[g], prr = g + 1 < n ? posc[g + 1] : posc[g];
				p = (int32_t)((u32)(prr - pl) * (u32)cv[i]);
			}
			pr[i] = p;
		}
		BLOCK_SYNC();
		const int cnt = block_excl_scan(f, LB_TILE);
		const int psum = block_excl_scan(pr, LB_TILE);
		int64_t o0, q0;
		lb_tile_prefix2(c, 1, 2, t, cnt, psum, &o0, &q0);
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x)
		{
			const int64_t g = g0 + i;
			if(g >= n || cv[i] <= 0) continue;
			const int64_t o = o0 + f[i];
			const int32_t pl = posc[g], prr = g + 1 < n ? posc[g + 1] : posc[g];
			seg_l[o] = pl; seg_r[o] = prr; seg_c[o] = cv[i];
			const int before = i > 0 ? cv[i - 1] : cv[LB_TILE];
			seg_head[o] = (g > 0 && before > 0) ? 0 : 1;
			seg_psum[o] = q0 + pr[i];
		}
		const bool last = t == n_tiles - 1;
		if(last && threadIdx.x == 0) { seg_psum[o0 + cnt] = q0 + psum; *n_seg = o0 + cnt; }
		// bundles whose first border falls into this tile (the last tile also owns rank n)
		const int64_t hi = last ? n + 1 : g0 + LB_TILE;
		for(int b = tile_b0[t] + (int)threadIdx.x; b <= n_bundles && bord_off[b] < hi; b += blockDim.x)
			seg_off[b] = o0 + f[bord_off[b] - g0];
		BLOCK_SYNC();
	}
}

// seg_nhead[o] = first segment after o that opens a run (n_seg if none), for the region walk of k_graph.h.  Tile t holds the
// segments n_seg - 1 - t * LB_TILE downwards (element k: segment top - k), so the next head of an element is the nearest head among
// the elements before it: an exclusive maximum scan of the heads' element indices.  What lies after the tile is found by reading
// the run heads that follow it until one is set -- runs are short (a run ends where the coverage drops to zero, at the latest at
// the end of the bundle), so tiles do not wait for each other.  The segment count stays on the device: the launch is sized by the
// border count, and tiles past the segments return at once.
#ifndef AGPU_EMU
#define NH_LANES 32
#else
#define NH_LANES 1               // kernel-logic build: one thread per CTA
#endif
KERNEL k_seg_nhead(int64_t n_bord, const uint8_t *seg_head, const int64_t *n_seg, int64_t *nhead)
{
	SHARED int s_tot[LB_ROW_TOTALS];
	SHARED long long s_after;
	const int64_t ns = *n_seg;
	const int64_t n_tiles = (n_bord + LB_TILE - 1) / LB_TILE;
	const auto mx = [](int x, int y) { return y > x ? y : x; };
	for(int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x)
	{
		const int64_t top = ns - 1 - t * LB_TILE;
		if(top < 0) break;
		// first head after the tile: warp 0 reads 8 x 32 run heads per step
		if(threadIdx.x < NH_LANES)
		{
			long long found = ns;
			for(int64_t p = top + 1; p < ns; p += 8 * NH_LANES)
			{
				u32 hit = 0;
				int r0 = 0;
#pragma unroll
				for(int r = 7; r >= 0; r--)
				{
					const int64_t q = p + r * NH_LANES + threadIdx.x;
					const bool on = q < ns && seg_head[q];
#ifndef AGPU_EMU
					const u32 m = __ballot_sync(0xffffffffu, on);
#else
					const u32 m = on ? 1u : 0u;
#endif
					if(m) { hit = m; r0 = r; }
				}
				if(hit) { found = p + r0 * NH_LANES + __ffs((int)hit) - 1; break; }
			}
			if(threadIdx.x == 0) s_after = found;
		}
		int h[LB_ROWS];
#pragma unroll
		for(int j = 0; j < LB_ROWS; j++)
		{
			const int k = j * LB_THREADS + threadIdx.x;
			h[j] = (top - k >= 0 && seg_head[top - k]) ? k : -1;
		}
		lb_rows_scan(h, -1, mx, s_tot);      // its barrier also publishes s_after
		const long long after = s_after;
#pragma unroll
		for(int j = 0; j < LB_ROWS; j++)
		{
			const int64_t s = top - (j * LB_THREADS + threadIdx.x);
			if(s >= 0) nhead[s] = h[j] >= 0 ? top - h[j] : after;
		}
		BLOCK_SYNC();
	}
}

// ---- CIGAR walk by warps: the walks for batches of long CIGARs (long reads: tens of operations per hit) ----------------------
// The thread-per-hit walks above read a hit's operations one after the other (35 dependent iterations per hit at configs[4],
// every load a different cache line from its neighbour lanes' loads).  Here a warp takes a GROUP of 32 consecutive hits: lane j
// loads the fields of hit j (one coalesced load per field, one pass over the dependent bundle lookups for all 32), then the
// warp walks the hits one after the other, the fields of the current one broadcast by shuffles, its operations loaded 32 at a
// time by the lanes -- and the first 32 operations of the NEXT hit requested before the current one is processed, so a hit
// costs no load latency of its own (a first version with one hit per warp and its loads in front of the walk ran 4.9 + 4.2 ms
// at configs[4] against 6.0 + 3.7 ms for the thread-per-hit walks: ~3.5 us of dependent loads per hit and warp).  The reference
// position after every operation is pos + a warp scan of the reference-consuming lengths; the index of an inner N operation
// among the hit's splices and of an M operation among its match blocks (the skip mask of the insert-size preview) are ballot
// counts.  Selected per batch by the mean number of operations per hit (warp_min_ops() in aletsch_gpu.cu).
#ifndef AGPU_EMU
#define CW_WS 32
#else
#define CW_WS 1                  // kernel-logic build: a "warp" of one lane runs the same code on groups of one hit
#endif
#define CW_WARPS 8

DEV int cw_excl_scan(int v, int lane, int *total)
{
#ifndef AGPU_EMU
	int inc = v;
#pragma unroll
	for(int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, inc, o); if(lane >= o) inc += y; }
	*total = __shfl_sync(0xffffffffu, inc, 31);
	return inc - v;
#else
	(void)lane;
	*total = v;
	return 0;
#endif
}
DEV u32 cw_ballot(bool p)
{
#ifndef AGPU_EMU
	return __ballot_sync(0xffffffffu, p);
#else
	return p ? 1u : 0u;
#endif
}
template<typename T> DEV T cw_shfl(T v, int j)
{
#ifndef AGPU_EMU
	return __shfl_sync(0xffffffffu, v, j);
#else
	(void)j;
	return v;
#endif
}

// the walk of one group: begin(j) before hit j, chunk(j, first, k, c0, c1, act, op, len, pe) for every 32 operations (pe = the
// reference position after the lane's operation), end(j, p) with the position after the last one.  All hooks run warp-uniformly.
template<typename B, typename C, typename E> DEV void cw_walk(const hits_dev &h, int64_t g, int lane, B begin, C chunk, E end)
{
	const int64_t i = g * CW_WS + lane;
	const bool valid = i < h.n_hits;
	const u32 c0 = valid ? h.cigar_off[i] : 0u, c1 = valid ? h.cigar_off[i + 1] : 0u;
	const int32_t p0 = valid ? h.pos[i] : 0;
	const u32 f0 = cw_shfl(c0, 0), f1 = cw_shfl(c1, 0);
	u32 nxt = f0 + lane < f1 ? h.cigar[f0 + lane] : 0u;
	for(int j = 0; j < CW_WS; j++)
	{
		const u32 jc0 = cw_shfl(c0, j), jc1 = cw_shfl(c1, j);
		int32_t p = cw_shfl(p0, j);
		u32 c = nxt;
		if(j + 1 < CW_WS)
		{
			const u32 n0 = cw_shfl(c0, j + 1), n1 = cw_shfl(c1, j + 1);
			nxt = n0 + lane < n1 ? h.cigar[n0 + lane] : 0u;
		}
		begin(j);
		for(u32 k0 = jc0; k0 < jc1; k0 += CW_WS)
		{
			const u32 k = k0 + lane;
			const bool act = k < jc1;
			if(k0 != jc0) c = act ? h.cigar[k] : 0u;
			const u32 op = c & 0xf, len = c >> 4;
			const int adv = (act && ((0x3C1A7 >> (op << 1)) & 2)) ? (int)len : 0;      // bam_cigar_type: consumes reference
			int tot;
			const int32_t pe = p + cw_excl_scan(adv, lane, &tot) + adv;
			chunk(j, k0 == jc0, k, jc0, jc1, act, op, len, pe);
			p += tot;
		}
		end(j, p);
	}
}

KERNEL k_hit_cigar_warp(hits_dev h, const int32_t *b_lpos, const int64_t *cov_base, u32 *border,
		int32_t *spl, int32_t *hit_nspl, const int32_t *hit_bundle, int32_t *n_spliced, int *err, const uint16_t *skip)
{
	const int lane = threadIdx.x % CW_WS, warp = threadIdx.x / CW_WS;
	const int wpb = blockDim.x / CW_WS;
	const u32 lt = (1u << lane) - 1u;
	const int64_t n_groups = (h.n_hits + CW_WS - 1) / CW_WS;
	for(int64_t g = (int64_t)blockIdx.x * wpb + warp; g < n_groups; g += (int64_t)gridDim.x * wpb)
	{
		const int64_t i = g * CW_WS + lane;
		const bool valid = i < h.n_hits;
		const int b = valid ? hit_bundle[i] : -1;
		const int64_t wb = valid ? cov_base[b] - (int64_t)b_lpos[b] : 0;
		const u32 sk = (valid && skip) ? skip[i] : 0u;
		const int32_t rp = valid ? h.rpos[i] : 0;
		int my_ns = 0;
		int32_t my_p = 0;
		int64_t jwb = 0;
		u32 jsk = 0;
		int z = 0, ns = 0;
		cw_walk(h, g, lane,
			[&](int j) { jwb = cw_shfl(wb, j); jsk = cw_shfl(sk, j); z = 0; ns = 0; },
			[&](int, bool, u32 k, u32 jc0, u32 jc1, bool act, u32 op, u32 len, int32_t pe)
			{
				const bool isM = act && op == 0;                                           // BAM_CMATCH
				const u32 mM = cw_ballot(isM);
				const int zi = z + __popc(mM & lt);
				if(isM && len > 0 && !(zi < 16 && ((jsk >> zi) & 1u)))
				{
					border_set(border, jwb + pe - (int32_t)len);
					border_set(border, jwb + pe);
				}
				const bool isN = act && op == 3 && k != jc0 && k != jc1 - 1;               // BAM_CREF_SKIP, not first / last op
				const u32 mN = cw_ballot(isN);
				if(isN)
				{
					int32_t *out = spl + jc0 + ns + 2 * __popc(mN & lt);
					out[0] = pe - (int32_t)len;
					out[1] = pe;
				}
				z += __popc(mM); ns += 2 * __popc(mN);
			},
			[&](int j, int32_t p) { if(lane == j) { my_ns = ns; my_p = p; } });
		if(valid)
		{
			if(my_p != rp) atomicAdd(&err[ERR_RPOS], 1);
			hit_nspl[i] = my_ns;
		}
#ifndef AGPU_EMU
		// the lanes hold consecutive hits: one atomic per (warp, bundle) instead of one per spliced hit
		const unsigned peers = __match_any_sync(0xffffffffu, (valid && my_ns > 0) ? b : -1);
		if(valid && my_ns > 0 && lane == __ffs((int)peers) - 1) atomicAdd(&n_spliced[b], __popc(peers));
#else
		if(valid && my_ns > 0) atomicAdd(&n_spliced[b], 1);
#endif
	}
}

KERNEL k_cov_add_warp(hits_dev h, const int32_t *hit_bundle, const int32_t *b_lpos, const int64_t *cov_base, const u32 *border,
		const u32 *wrank, int32_t *diffc, const uint16_t *skip)
{
	const int lane = threadIdx.x % CW_WS, warp = threadIdx.x / CW_WS;
	const int wpb = blockDim.x / CW_WS;
	const u32 lt = (1u << lane) - 1u;
	const int64_t n_groups = (h.n_hits + CW_WS - 1) / CW_WS;
	for(int64_t g = (int64_t)blockIdx.x * wpb + warp; g < n_groups; g += (int64_t)gridDim.x * wpb)
	{
		const int64_t i = g * CW_WS + lane;
		const bool valid = i < h.n_hits;
		const int b = valid ? hit_bundle[i] : -1;
		const int64_t wb = valid ? cov_base[b] - (int64_t)b_lpos[b] : 0;
		const u32 sk = (valid && skip) ? skip[i] : 0u;
		int64_t jwb = 0;
		u32 jsk = 0;
		int z = 0;
		cw_walk(h, g, lane,
			[&](int j) { jwb = cw_shfl(wb, j); jsk = cw_shfl(sk, j); z = 0; },
			[&](int, bool, u32, u32, u32, bool act, u32 op, u32 len, int32_t pe)
			{
				const bool isM = act && op == 0;
				const u32 mM = cw_ballot(isM);
				const int zi = z + __popc(mM & lt);
				if(isM && len > 0 && !(zi < 16 && ((jsk >> zi) & 1u)))
				{
					atomicAdd(&diffc[border_rank(border, wrank, jwb + pe - (int32_t)len)], 1);
					atomicAdd(&diffc[border_rank(border, wrank, jwb + pe)], -1);
				}
				z += __popc(mM);
			},
			[&](int, int32_t) {});
	}
}

// hit.rpos = pos + bam_cigar2rlen (rnacore/hit.cc:64)
KERNEL k_hit_rpos_warp(hits_dev h, int32_t *rpos)
{
	const int lane = threadIdx.x % CW_WS, warp = threadIdx.x / CW_WS;
	const int wpb = blockDim.x / CW_WS;
	const int64_t n_groups = (h.n_hits + CW_WS - 1) / CW_WS;
	for(int64_t g = (int64_t)blockIdx.x * wpb + warp; g < n_groups; g += (int64_t)gridDim.x * wpb)
	{
		const int64_t i = g * CW_WS + lane;
		int32_t my_p = 0;
		cw_walk(h, g, lane, [&](int) {}, [&](int, bool, u32, u32, u32, bool, u32, u32, int32_t) {},
			[&](int j, int32_t p) { if(lane == j) my_p = p; });
		if(i < h.n_hits) rpos[i] = my_p;
	}
}

// extra coverage intervals of a bundle (insert-size preview: runs of earlier bundles flushed into this one): clipped to the bundle's
// window [lpos, covhi], a border bit at either end and a weighted point each (k_cov_add_points adds them by rank); intervals that
// miss the window get weight 0
KERNEL k_extra_intervals(int64_t n, const int32_t *ex_bundle, const int32_t *ex_l, const int32_t *ex_r, const int32_t *ex_cnt, const int32_t *b_lpos,
		const int32_t *b_covhi, const int64_t *cov_base, u32 *border, int64_t *pt_g, int32_t *pt_d)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n) return;
	const int b = ex_bundle[i];
	int32_t l = ex_l[i], r = ex_r[i];
	if(l < b_lpos[b]) l = b_lpos[b];
	if(r > b_covhi[b]) r = b_covhi[b];
	pt_g[2 * i] = cov_base[b]; pt_g[2 * i + 1] = cov_base[b];
	pt_d[2 * i] = 0; pt_d[2 * i + 1] = 0;
	if(l >= r) return;
	const int64_t s = cov_base[b] + (l - b_lpos[b]), e = cov_base[b] + (r - b_lpos[b]);
	atomicOr(&border[s >> 5], 1u << (s & 31));
	atomicOr(&border[e >> 5], 1u << (e & 31));
	pt_g[2 * i] = s; pt_d[2 * i] = ex_cnt[i];
	pt_g[2 * i + 1] = e; pt_d[2 * i + 1] = -ex_cnt[i];
}

} // namespace agpu




#endif
