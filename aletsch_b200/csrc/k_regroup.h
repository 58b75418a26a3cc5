// Regrouping of bundles that already sit in HBM (agpu_batch_gather): a new batch whose bundle k is bundle sel_bundle[k] of source
// sel_src[k].  A streaming copy with no counterpart in the reference: it lets the cross-sample stages cut a job a second time,
// by cluster instead of by position, without sending the hits over PCIe again (aletsch_b200/clusters.py).
//
// Sizes: one thread per selected bundle; two device-wide scans turn them into the output's bundle_hit_off and the CIGAR base of
// every bundle.  Hits and CIGAR words are then copied balanced over the OUTPUT elements (bundle sizes are skewed: one CTA per
// bundle would leave the copy waiting for the deepest one); an element finds its bundle by the one-bisection-per-tile scheme of
// k_tile_bundle (k_evidence.h).
#ifndef ALETSCH_B200_CSRC_K_REGROUP_H
#define ALETSCH_B200_CSRC_K_REGROUP_H

#include "dev.h"
#include "k_evidence.h"

namespace agpu {

// per selected bundle: hits, CIGAR operations, and where both start in the source
KERNEL k_gather_sizes(int32_t n_sel, const hits_dev *src, const int32_t *sel_src, const int32_t *sel_bundle, int64_t *n_hit, int64_t *n_op,
		int64_t *src_h0, int64_t *src_c0)
{
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	if(k >= n_sel) return;
	const hits_dev &s = src[sel_src[k]];
	const int b = sel_bundle[k];
	const int64_t h0 = s.bundle_hit_off[b], h1 = s.bundle_hit_off[b + 1];
	const int64_t c0 = s.cigar_off[h0];
	n_hit[k] = h1 - h0;
	n_op[k] = (int64_t)s.cigar_off[h1] - c0;
	src_h0[k] = h0;
	src_c0[k] = c0;
}

// selected bundle of the first element of every tile of HB_TILE output elements (hits or CIGAR words) under the offsets off[]
KERNEL k_gather_tiles(const int64_t *off, int32_t n_sel, int64_t n, int64_t n_tiles, int32_t *tile)
{
	const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(t > n_tiles) return;
	const int64_t i = t * HB_TILE;
	tile[t] = i < n ? bundle_of_hit(off, 0, n_sel, i) : n_sel - 1;
}

DEV int gather_bundle(const int64_t *off, const int32_t *tile, int64_t i)
{
	const int64_t t = i / HB_TILE;
	const int lo = tile[t], hi = tile[t + 1];
	return lo == hi ? lo : bundle_of_hit(off, lo, hi + 1, i);
}

// one thread per output hit: the six per-hit arrays, the strand (per hit, or the bundle's strand expanded), and cigar_off rebased to
// the output's CIGAR base of the bundle.  Thread n_hits writes cigar_off[n_hits] = the CIGAR total.
KERNEL k_gather_hits(int64_t n_hits, int32_t n_sel, const hits_dev *src, const int32_t *sel_src, const int32_t *sel_bundle, const int64_t *hit_off,
		const int32_t *tile, const int64_t *src_h0, const int64_t *src_c0, const int64_t *op_off,
		int32_t *pos, int32_t *rpos, int32_t *mpos, int32_t *isize, uint8_t *strand, uint8_t *xs, u64 *qid, u32 *cigar_off)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i > n_hits) return;
	if(i == n_hits) { cigar_off[i] = (u32)op_off[n_sel]; return; }
	const int k = gather_bundle(hit_off, tile, i);
	const hits_dev &s = src[sel_src[k]];
	const int64_t j = src_h0[k] + (i - hit_off[k]);
	pos[i] = s.pos[j]; rpos[i] = s.rpos[j]; mpos[i] = s.mpos[j]; isize[i] = s.isize[j];
	xs[i] = s.xs[j]; qid[i] = s.qid[j];
	strand[i] = s.strand ? s.strand[j] : s.bundle_strand[sel_bundle[k]];
	cigar_off[i] = (u32)(op_off[k] + ((int64_t)s.cigar_off[j] - src_c0[k]));
}

// one thread per output CIGAR word: every selected bundle's operations are one contiguous run of its source
KERNEL k_gather_cigar(int64_t n_ops, const hits_dev *src, const int32_t *sel_src, const int64_t *op_off, const int32_t *tile, const int64_t *src_c0,
		u32 *cigar)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_ops) return;
	const int k = gather_bundle(op_off, tile, i);
	cigar[i] = src[sel_src[k]].cigar[src_c0[k] + (i - op_off[k])];
}

} // namespace agpu

#endif
