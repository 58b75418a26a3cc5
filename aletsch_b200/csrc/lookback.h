// Single-pass device-wide prefix sums (decoupled look-back): every device-wide scan of the path is ONE launch instead of the
// tile-sum / single-CTA scan / apply triple.
//
// A CTA takes the next tile from a ticket counter (tiles are therefore started in index order, which is what makes waiting for
// a predecessor safe), scans it in shared memory, publishes the tile's aggregate in a 64-bit status word, then walks back over
// its predecessors' words until it meets one that already holds an inclusive prefix.  Status word:
//     [63:62] 0 = nothing yet, 1 = tile aggregate, 2 = inclusive prefix   [61:48] launch epoch   [47:0] value (two's complement)
// The epoch makes words of earlier launches read as "nothing yet", so the status array is never cleared between launches; the
// ticket counter is never reset either: every launch consumes exactly n_tiles + gridDim.x tickets and the host passes the
// running total (lb_launch below).  Values are exact up to 2^47 in magnitude.
//
// Kernel-logic test build: CTAs run one after the other with blockDim.x == 1, so the first "CTA" takes every ticket in order
// and every look-back finds its predecessor complete.
#ifndef ALETSCH_B200_CSRC_LOOKBACK_H
#define ALETSCH_B200_CSRC_LOOKBACK_H

#include "dev.h"
#include "blockops.h"

namespace agpu {

#define LB_TILE 2048
#define LB_AGG 1ULL
#define LB_INC 2ULL
#define LB_CHAINS 4              // independent status arrays a kernel may chain (e.g. coverage sum -> segment count -> product sum)

// what a look-back kernel needs from the host: status words of LB_CHAINS chains of `stride` tiles each, the ticket counter, this
// launch's epoch and the tickets consumed before it
struct lb_ctl
{
	u64 *status;
	unsigned long long *ticket;
	int64_t stride;
	unsigned long long ticket_base;
	u32 epoch;
};

HD u64 lb_pack(u64 flag, u32 epoch, int64_t v) { return (flag << 62) | ((u64)(epoch & 0x3fffu) << 48) | ((u64)v & 0xffffffffffffULL); }
HD int64_t lb_value(u64 w) { return ((int64_t)(w << 16)) >> 16; }

DEV u64 lb_load(const u64 *p)
{
#ifndef AGPU_EMU
	return *(const volatile u64*)p;
#else
	return *p;
#endif
}
DEV void lb_store(u64 *p, u64 w)
{
#ifndef AGPU_EMU
	*(volatile u64*)p = w;
#else
	*p = w;
#endif
}

// next tile of this launch for the CTA, or -1 when the launch is exhausted (all threads get the same answer)
DEV int64_t lb_next_tile(const lb_ctl &c, int64_t n_tiles)
{
	SHARED long long s_tile;
	BLOCK_SYNC();
	if(threadIdx.x == 0)
	{
		unsigned long long t = atomicAdd(c.ticket, 1ULL) - c.ticket_base;
		s_tile = t < (unsigned long long)n_tiles ? (long long)t : -1;
	}
	BLOCK_SYNC();
	return (int64_t)s_tile;
}

// called by ONE thread of the CTA: publish the aggregate of `tile` on chain `chain`, return the sum of all earlier tiles
DEV int64_t lb_resolve(const lb_ctl &c, int chain, int64_t tile, int64_t aggregate)
{
	u64 *st = c.status + (int64_t)chain * c.stride;
	if(tile == 0) { lb_store(&st[0], lb_pack(LB_INC, c.epoch, aggregate)); return 0; }
	lb_store(&st[tile], lb_pack(LB_AGG, c.epoch, aggregate));
	int64_t run = 0;
	int64_t p = tile - 1;
	while(true)
	{
		const u64 w = lb_load(&st[p]);
		const u64 flag = w >> 62;
		if(flag == 0 || ((u32)(w >> 48) & 0x3fffu) != (c.epoch & 0x3fffu)) continue;      // not published in this launch yet
		run += lb_value(w);
		if(flag == LB_INC) break;
		p--;
	}
	lb_store(&st[tile], lb_pack(LB_INC, c.epoch, run + aggregate));
	return run;
}

#ifndef AGPU_EMU
// the same by the 32 lanes of ONE warp: the window of the 32 nearest predecessors is read at once, so a tile whose
// predecessors only hold aggregates yet walks back 32 tiles per round trip to L2 instead of one (a launch starts with ~1200
// tiles in flight and nothing but tile 0 inclusive: the one-thread walk made a scan of 6 M values take 55 us, 1.4 TB/s)
__device__ int64_t lb_resolve_warp(const lb_ctl &c, int chain, int64_t tile, int64_t aggregate)
{
	const unsigned FULL = 0xffffffffu;
	const int lane = threadIdx.x & 31;
	u64 *st = c.status + (int64_t)chain * c.stride;
	if(tile == 0) { if(lane == 0) lb_store(&st[0], lb_pack(LB_INC, c.epoch, aggregate)); return 0; }
	if(lane == 0) lb_store(&st[tile], lb_pack(LB_AGG, c.epoch, aggregate));
	int64_t run = 0;
	int64_t p = tile - 1;
	while(true)
	{
		const int64_t idx = p - lane;
		u64 flag = LB_INC;                    // in front of tile 0: an inclusive prefix of 0
		int64_t val = 0;
		if(idx >= 0)
		{
			const u64 w = lb_load(&st[idx]);
			flag = w >> 62;
			if(((u32)(w >> 48) & 0x3fffu) != (c.epoch & 0x3fffu)) flag = 0;      // a word of an earlier launch
			val = lb_value(w);
		}
		const unsigned inc = __ballot_sync(FULL, flag == LB_INC), missing = __ballot_sync(FULL, flag == 0);
		const int first = inc ? __ffs((int)inc) - 1 : 32;                       // the nearest inclusive prefix in the window
		const unsigned need = first >= 31 ? FULL : ((2u << first) - 1u);          // lanes 0 .. first
		if(missing & need) continue;                                             // not all published yet: read the window again
		int64_t v = lane <= first ? val : 0;
#pragma unroll
		for(int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
		run += v;
		if(inc) break;
		p -= 32;
	}
	if(lane == 0) lb_store(&st[tile], lb_pack(LB_INC, c.epoch, run + aggregate));
	return run;
}
#endif

// CTA-wide: exclusive prefix of the tile on `chain` broadcast to every thread (aggregate must be the same in all threads)
DEV int64_t lb_tile_prefix(const lb_ctl &c, int chain, int64_t tile, int64_t aggregate)
{
	SHARED long long s_pre[LB_CHAINS];
#ifndef AGPU_EMU
	if(blockDim.x >= 32)
	{
		if(threadIdx.x < 32) { const int64_t r = lb_resolve_warp(c, chain, tile, aggregate); if(threadIdx.x == 0) s_pre[chain] = r; }
	}
	else
#endif
	if(threadIdx.x == 0) s_pre[chain] = lb_resolve(c, chain, tile, aggregate);
	BLOCK_SYNC();
	return (int64_t)s_pre[chain];
}

// the same for two chains whose aggregates are known together: resolved side by side by two warps, one barrier
DEV void lb_tile_prefix2(const lb_ctl &c, int chain_a, int chain_b, int64_t tile, int64_t agg_a, int64_t agg_b, int64_t *pre_a, int64_t *pre_b)
{
	SHARED long long s_pre2[2];
#ifndef AGPU_EMU
	if(blockDim.x >= 64)
	{
		const int w = threadIdx.x >> 5;
		if(w < 2)
		{
			const int64_t r = lb_resolve_warp(c, w ? chain_b : chain_a, tile, w ? agg_b : agg_a);
			if((threadIdx.x & 31) == 0) s_pre2[w] = r;
		}
	}
	else
#endif
	if(threadIdx.x == 0) { s_pre2[0] = lb_resolve(c, chain_a, tile, agg_a); s_pre2[1] = lb_resolve(c, chain_b, tile, agg_b); }
	BLOCK_SYNC();
	*pre_a = (int64_t)s_pre2[0];
	*pre_b = (int64_t)s_pre2[1];
}

// ---- tiles held in registers: thread t owns the elements t, t + LB_THREADS, t + 2 LB_THREADS, ... of the tile (LB_ROWS of them,
// every global access of a row coalesced).  lb_rows_scan turns them into exclusive prefixes in tile order with warp shuffles;
// the (row, warp) totals go through shared memory once, so a scan costs one barrier and no bank conflicts.
#ifndef AGPU_EMU
#define LB_THREADS 256           // the CTA of LAUNCH_LB
#else
#define LB_THREADS 1             // kernel-logic build: one thread per CTA owns the whole tile
#endif
#define LB_ROWS (LB_TILE / LB_THREADS)
#define LB_ROW_TOTALS (LB_ROWS * LB_THREADS / 32 + 1)

// v[j] <- combine of the tile's elements before element j of this thread; returns the combine of the whole tile.  `s_tot`: shared
// scratch of LB_ROW_TOTALS values, not reused before the next barrier.  The values of one scan are combined in a different order
// than an element-by-element loop, so `op` must be associative and commutative; int sums wrap (compute them as unsigned).
template<typename T, typename Op> DEV T lb_rows_scan(T (&v)[LB_ROWS], T ident, Op op, T *s_tot)
{
#ifndef AGPU_EMU
	static_assert(LB_ROWS * LB_THREADS / 32 == 64, "lb_rows_scan: 64 (row, warp) totals");
	const unsigned FULL = 0xffffffffu;
	const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	const int NW = LB_THREADS / 32;
	T ex[LB_ROWS];
#pragma unroll
	for(int j = 0; j < LB_ROWS; j++)
	{
		T inc = v[j];
#pragma unroll
		for(int o = 1; o < 32; o <<= 1) { const T y = __shfl_up_sync(FULL, inc, o); if(lane >= o) inc = op(y, inc); }
		const T up = __shfl_up_sync(FULL, inc, 1);
		ex[j] = lane > 0 ? up : ident;
		if(lane == 31) s_tot[j * NW + w] = inc;
	}
	__syncthreads();
	// exclusive prefixes of the 64 totals in (row, warp) order, by every warp: lane l holds totals l and 32 + l
	T a = s_tot[lane], b = s_tot[32 + lane];
#pragma unroll
	for(int o = 1; o < 32; o <<= 1)
	{
		const T ya = __shfl_up_sync(FULL, a, o), yb = __shfl_up_sync(FULL, b, o);
		if(lane >= o) { a = op(ya, a); b = op(yb, b); }
	}
	const T ta = __shfl_sync(FULL, a, 31), tb = __shfl_sync(FULL, b, 31);
	T ea = __shfl_up_sync(FULL, a, 1), eb = __shfl_up_sync(FULL, b, 1);
	if(lane == 0) { ea = ident; eb = ident; }
	eb = op(ta, eb);
#pragma unroll
	for(int j = 0; j < LB_ROWS; j++)
	{
		const int e = j * NW + w;                 // j * NW < 32 decides the half at compile time (j is unrolled, w < NW)
		const T p = j * NW < 32 ? __shfl_sync(FULL, ea, e & 31) : __shfl_sync(FULL, eb, e & 31);
		v[j] = op(p, ex[j]);
	}
	return op(ta, tb);
#else
	(void)s_tot;
	T run = ident;
	for(int j = 0; j < LB_ROWS; j++) { const T x = v[j]; v[j] = run; run = op(run, x); }
	return run;
#endif
}

// ---- generic scans ---------------------------------------------------------------------------------------------------------
// exclusive prefix sum of int32 values (mode 0) or of the flags (v[i] >= 0) (mode 1) into int64: out[i], out[n] = total
KERNEL k_lb_scan_i32(lb_ctl c, const int32_t *v, int64_t n, int mode, int64_t *out)
{
	SHARED16 int f[LB_TILE];
	const int64_t n_tiles = (n + 1 + LB_TILE - 1) / LB_TILE;
	for(int64_t t = lb_next_tile(c, n_tiles); t >= 0; t = lb_next_tile(c, n_tiles))
	{
		const int64_t g0 = t * LB_TILE;
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x)
		{
			const int64_t g = g0 + i;
			f[i] = g < n ? (mode ? (v[g] >= 0 ? 1 : 0) : v[g]) : 0;
		}
		BLOCK_SYNC();
		const int tot = block_excl_scan(f, LB_TILE);
		const int64_t pre = lb_tile_prefix(c, 0, t, tot);
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x)
		{
			const int64_t g = g0 + i;
			if(g <= n) out[g] = pre + f[i];
		}
	}
}

// the same over int64 values
KERNEL k_lb_scan_i64(lb_ctl c, const int64_t *v, int64_t n, int64_t *out)
{
	SHARED long long f[LB_TILE];
	SHARED long long part[AGPU_MAX_BLOCK];
	const int64_t n_tiles = (n + 1 + LB_TILE - 1) / LB_TILE;
	for(int64_t t = lb_next_tile(c, n_tiles); t >= 0; t = lb_next_tile(c, n_tiles))
	{
		const int64_t g0 = t * LB_TILE;
		const int nt = blockDim.x, th = threadIdx.x;
		const int chunk = (LB_TILE + nt - 1) / nt;
		int lo = th * chunk, hi = lo + chunk;
		if(lo > LB_TILE) lo = LB_TILE;
		if(hi > LB_TILE) hi = LB_TILE;
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x) { const int64_t g = g0 + i; f[i] = g < n ? v[g] : 0; }
		BLOCK_SYNC();
		long long sm = 0;
		for(int i = lo; i < hi; i++) sm += f[i];
		long long tot = 0, mine = 0;
#ifndef AGPU_EMU
		if((nt & 31) == 0)
		{
			// scan of the thread sums: warp shuffles, the warp totals through shared memory
			const int lane = th & 31, w = th >> 5, nw = nt >> 5;
			long long inc = sm;
#pragma unroll
			for(int o = 1; o < 32; o <<= 1) { long long y = __shfl_up_sync(0xffffffffu, inc, o); if(lane >= o) inc += y; }
			if(lane == 31) part[w] = inc;
			BLOCK_SYNC();
			long long pre = 0;
			for(int k = 0; k < nw; k++) { const long long s = part[k]; if(k < w) pre += s; tot += s; }
			mine = pre + inc - sm;
		}
		else
#endif
		{
			part[th] = sm;
			BLOCK_SYNC();
			for(int k = 0; k < nt; k++) { if(k == th) mine = tot; tot += part[k]; }
		}
		const int64_t pre = lb_tile_prefix(c, 0, t, tot);
		long long run = pre + mine;
		for(int i = lo; i < hi; i++) { const long long x = f[i]; f[i] = run; run += x; }
		BLOCK_SYNC();
		for(int i = threadIdx.x; i < LB_TILE; i += blockDim.x) { const int64_t g = g0 + i; if(g <= n) out[g] = f[i]; }
	}
}

// ---- per-bundle sized arrays (a few 10^4 elements): one CTA of 512 threads, no look-back machinery.  Thread t owns the
// elements t, t + 512, t + 1024, ... (coalesced rows); eight rows at a time are loaded into registers, so the global-memory
// latency is paid once per eight rows; every row is then scanned with warp shuffles and the 16 warp totals, with a running
// carry.  (A CTA that needs a whole SM's registers would starve next to the long kernels of the other streams of a pipeline.)
#define SMALL_SCAN_THREADS 512
#define SMALL_SCAN_RB 8
#define SMALL_SCAN_MAX 65536
template<typename T> DEV void small_scan(const T *in, int64_t n, int64_t *out)
{
#ifndef AGPU_EMU
	__shared__ long long wtot[2][32];
	const int t = threadIdx.x, lane = t & 31, w = t >> 5, nw = SMALL_SCAN_THREADS / 32;
	const int rows = (int)((n + SMALL_SCAN_THREADS - 1) / SMALL_SCAN_THREADS);
	long long carry = 0;
	int flip = 0;
	for(int r0 = 0; r0 < rows; r0 += SMALL_SCAN_RB)
	{
		long long v[SMALL_SCAN_RB];
#pragma unroll
		for(int k = 0; k < SMALL_SCAN_RB; k++) { const int64_t i = (int64_t)(r0 + k) * SMALL_SCAN_THREADS + t; v[k] = (r0 + k < rows && i < n) ? (long long)in[i] : 0; }
#pragma unroll
		for(int k = 0; k < SMALL_SCAN_RB; k++)
		{
			if(r0 + k >= rows) break;
			long long inc = v[k];
#pragma unroll
			for(int o = 1; o < 32; o <<= 1) { long long y = __shfl_up_sync(0xffffffffu, inc, o); if(lane >= o) inc += y; }
			if(lane == 31) wtot[flip][w] = inc;
			__syncthreads();
			long long x = lane < nw ? wtot[flip][lane] : 0, xi = x;
#pragma unroll
			for(int o = 1; o < 32; o <<= 1) { long long y = __shfl_up_sync(0xffffffffu, xi, o); if(lane >= o) xi += y; }
			const long long wpre = __shfl_sync(0xffffffffu, xi - x, w), total = __shfl_sync(0xffffffffu, xi, 31);
			const int64_t i = (int64_t)(r0 + k) * SMALL_SCAN_THREADS + t;
			if(i < n) out[i] = carry + wpre + inc - v[k];
			carry += total;
			flip ^= 1;
		}
	}
	if(t == 0) out[n] = carry;
#else
	if(threadIdx.x != 0) return;
	long long run = 0;
	for(int64_t i = 0; i < n; i++) { out[i] = run; run += (long long)in[i]; }
	out[n] = run;
#endif
}
#ifndef AGPU_EMU
#define SMALL_SCAN_KERNEL __global__ void __launch_bounds__(SMALL_SCAN_THREADS)
#else
#define SMALL_SCAN_KERNEL KERNEL
#endif
SMALL_SCAN_KERNEL k_small_scan_i32(const int32_t *in, int64_t n, int64_t *out) { small_scan<int32_t>(in, n, out); }
SMALL_SCAN_KERNEL k_small_scan_i64(const int64_t *in, int64_t n, int64_t *out) { small_scan<int64_t>(in, n, out); }
// up to 8 arrays of the same length in one launch, one CTA each (the five per-bundle bounds of the graph stage, the two job
// counts of the bridging stage: every launch saved is ~20 us of a serial chain)
struct small_scan_set { const int64_t *in[8]; int64_t *out[8]; };
SMALL_SCAN_KERNEL k_small_scan_i64_multi(small_scan_set s, int64_t n) { small_scan<int64_t>(s.in[blockIdx.x], n, s.out[blockIdx.x]); }

} // namespace agpu

#endif
