// libaletsch_gpu.so: implementation of include/aletsch_gpu.h.
// Compiled by nvcc for sm_100a (product) or, for the CPU-only kernel-logic tests, by g++ with
// -DAGPU_EMU (tests/emu; never shipped, see dev.h).
#include "runtime.h"
#include "k_evidence.h"
#include "k_graph.h"
#include "k_fragments.h"
#include "k_cluster.h"
#include "k_bridge.h"
#include "k_similarity.h"
#include "k_group.h"
#include "k_phase.h"
#include "k_revise.h"
#include "k_support.h"
#include "k_unpack.h"
#include "k_fetch.h"
#include "k_regroup.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <map>
#include <new>
#include <thread>

#ifdef AGPU_EMU
thread_local agpu_emu_dim threadIdx, blockIdx, blockDim, gridDim;
// marks the emulation build for its callers: its "device" pointers (agpu_batch_inputs) are host memory
extern "C" const int agpu_emu_build = 1;
#endif

using namespace agpu;

// ------------------------------------------------------------------------------------------
// device chain_set (hcst / fcst)
struct chainset_state
{
	bool built = false;
	int64_t n_elem = 0;
	const int64_t *d_elem_off = NULL;     // [NB+1]
	const int32_t *val = NULL;
	const u32 *voff32 = NULL;
	const int64_t *voff64 = NULL;
	const int32_t *elem_len = NULL;
	dbuf<int64_t> reg_off, elem_slot, c_slot, val_base;
	dbuf<u64> slot_word, key_scratch, key_scratch2;
	dbuf<int32_t> slot_first, slot_cnt, slot_chain, n_chains, n_splices, c_rep, c_cnt, c_grp, handle_chain, splices_scratch;
	int64_t n_slots = 0;
	// combined chain sets (k_group.h) own their element arrays: coordinates offset / length / AI3 counts per element and the
	// element offsets per combined bundle
	dbuf<int64_t> ext_voff, ext_goff;
	dbuf<int32_t> ext_len, ext_cnt3, ext_val;
	std::vector<int64_t> ext_goff_host;
	int64_t ext_nval = 0;                 // size of the (shared) coordinate array `val` points into

	chains_view view() const
	{
		chains_view v;
		v.present = built ? 1 : 0;
		v.elem_off = d_elem_off; v.n_chains = n_chains.p; v.c_rep = c_rep.p; v.c_cnt = c_cnt.p;
		v.elem_len = elem_len; v.voff32 = voff32; v.voff64 = voff64; v.val = val;
		return v;
	}
};

struct graph_state
{
	bool built = false;
	dbuf<int64_t> ub[5], off[5];
	int64_t tot[5] = {0, 0, 0, 0, 0};
	dbuf<int32_t> iarena;
	dbuf<u64> karena;
	dbuf<int32_t> n_junc, n_pex, n_edge;
	dbuf<int32_t> j[9];
	dbuf<int32_t> p_i[6];
	dbuf<double> p_d[3];
	dbuf<int32_t> v_i[6];
	dbuf<double> v_d[3];
	dbuf<int32_t> e_i[3];
	dbuf<double> e_w;
	dbuf<int32_t> in_off, in_src, in_eid, out_off, out_dst, out_eid;

	graph_dev dev(int *err) const
	{
		graph_dev g;
		g.junc_off = off[0].p; g.pex_off = off[1].p; g.edge_off = off[2].p; g.iarena_off = off[3].p; g.karena_off = off[4].p;
		g.iarena = iarena.p; g.karena = karena.p;
		g.n_junc = n_junc.p; g.n_pex = n_pex.p; g.n_edge = n_edge.p;
		g.j_l = j[0].p; g.j_r = j[1].p; g.j_cnt = j[2].p; g.j_xs0 = j[3].p; g.j_xs1 = j[4].p; g.j_xs2 = j[5].p;
		g.j_strand = j[6].p; g.j_lexon = j[7].p; g.j_rexon = j[8].p;
		g.p_l = p_i[0].p; g.p_r = p_i[1].p; g.p_lt = p_i[2].p; g.p_rt = p_i[3].p; g.p_regional = p_i[4].p; g.p_type = p_i[5].p;
		g.p_ave = p_d[0].p; g.p_dev = p_d[1].p; g.p_max = p_d[2].p;
		g.v_l = v_i[0].p; g.v_r = v_i[1].p; g.v_len = v_i[2].p; g.v_type = v_i[3].p; g.v_regional = v_i[4].p; g.v_brk = v_i[5].p;
		g.v_w = v_d[0].p; g.v_dev = v_d[1].p; g.v_max = v_d[2].p;
		g.e_s = e_i[0].p; g.e_t = e_i[1].p; g.e_strand = e_i[2].p; g.e_w = e_w.p;
		g.in_off = in_off.p; g.in_src = in_src.p; g.in_eid = in_eid.p;
		g.out_off = out_off.p; g.out_dst = out_dst.p; g.out_eid = out_eid.p;
		g.remap = NULL;
		g.err = err;
		return g;
	}
};

// cross-sample support features (k_support.h): the graphs of all cluster members + combined graphs in one layout, and the result rows
struct support_state
{
	bool built = false;
	int32_t n_groups = 0, n_members = 0;
	int64_t n_vert = 0, n_ecap = 0, nnz = 0;
	dbuf<int64_t> voff, eoff, row_off;
	dbuf<int32_t> ne, vl, vr, out_off, in_off, in_eid, es, et, count, row_slot;
	dbuf<double> vwA, vwB, ewA, ewB, abd, loss, row_val;
	dbuf<uint8_t> aliveB;
	std::vector<int32_t> ne_host, slot_off_host, slot_sample_host, member_group_host;
};

// everything the stages derive from a batch's input: agpu_batch_reset drops it by assigning a default-constructed one
struct batch_derived
{
	// evidence
	bool evidence = false;
	dbuf<int32_t> b_lpos, b_rpos, b_covhi;
	dbuf<uint8_t> b_strand;
	dbuf<int64_t> b_span, cov_base;
	int64_t ltot = 0;
	// coverage map on border-compacted coordinates (k_evidence.h, coverage section)
	dbuf<u32> border, wrank;
	dbuf<int32_t> diffc, posc;
	dbuf<int64_t> bord_off, ex_s, ex_e;
	int64_t n_bord = 0, n_extra = 0;
	// a combined bundle's coverage sources: the borders of its members as weighted window positions (k_group.h)
	dbuf<int64_t> pt_g;
	dbuf<int32_t> pt_d;
	int64_t n_pts = 0;
	dbuf<int32_t> spl, hit_nspl, hit_bundle;
	// insert-size preview result: fragment length per cluster (INT32_MIN: not counted)
	dbuf<int32_t> pv_isize;
	bool preview_built = false;
	chainset_state hcst, fcst;
	// segments
	bool cov_dirty = true;
	dbuf<int64_t> seg_off;
	dbuf<int32_t> seg_l, seg_r, seg_c;
	dbuf<int64_t> seg_nhead, seg_psum;     // run structure and prefix sums of len * cov over all segments (k_graph.h seg_view)
	dbuf<int64_t> cov_tot;                 // [0] borders, [1] segments
	int64_t n_seg = 0;
	bool n_seg_on_dev = false;             // n_seg is still to be read back from cov_tot (seg_count)

	// fragments / clusters / bridges live in their own headers' state structs
	fragments_state frg;
	graph_state gr;
	cluster_state clu;
	bridge_state brg;
	bridge_entries ent;

	// phasing paths (bundle_base::build_phase_set): distinct coordinate lists in element order + counts
	bool phase_built = false;
	int64_t n_phase = 0, n_phase_val = 0;
	dbuf<int32_t> ph_val, ph_len, ph_cnt;
	dbuf<int64_t> ph_off, ph_boff;
	// combined phase sets of bundle clusters (agpu_batch_group_phase_set): distinct lists per cluster in element order, their
	// coordinates in ph_val
	bool gphase_built = false;
	int32_t gph_ng = 0;
	int64_t n_gphase = 0;
	dbuf<int32_t> gph_len, gph_cnt;
	dbuf<int64_t> gph_off, gph_boff;

	// boundary revision (identify_boundaries / remove_false_boundaries): added edges and vertex annotations, in the vertex
	// layout of the graphs
	bool revise_built = false;
	dbuf<int32_t> rv_nstart, rv_nend, rv_addv, rv_leave, rv_come;
	dbuf<double> rv_addw, rv_lratio, rv_cratio;
	dbuf<int64_t> rv_voff;
	int64_t rv_nvert = 0;

	support_state sup;
	// group-level re-bridge (assembler::bridge): the combined bundles of the clusters as a batch of their own (freed with
	// agpu_batch_free)
	agpu_batch *cb = NULL;
	dbuf<int32_t> g_remap, g_members, g_first;
	dbuf<int64_t> g_member_off;
	std::vector<int32_t> g_order_host;     // members of every cluster in combine order (flattened like the input)
	bool group_pass = false;               // cluster / bridge stages work against cb's graphs
};

struct agpu_batch : batch_derived
{
	int32_t nb = 0;
	int64_t nh = 0, nc = 0;
	bool owns_input = false;
	hits_dev h;
	// owned copies of the input (upload path)
	dbuf<int64_t> in_hit_off;
	dbuf<int32_t> in_pos, in_rpos, in_mpos, in_isize;
	dbuf<uint16_t> in_flag;
	dbuf<uint8_t> in_strand, in_xs, in_bstrand;
	dbuf<u64> in_qid;
	dbuf<u32> in_cigar_off, in_cigar;
	std::vector<int64_t> hit_off_host;
	std::vector<int32_t> tid_host, sample_host;
	// bundles by descending hit count: [0, n_large) get wide CTAs, the rest one warp each
	dbuf<int32_t> order;
	int32_t n_large = 0;
	// regions of the per-bundle qname tables (mate pairing): a power of two >= 1.5 x the bundle's hits

	dbuf<int> err;

	// coverage edits of the insert-size preview (agpu_batch_coverage_edit): blocks without coverage, foreign intervals; part of the
	// batch's INPUT (kept across agpu_batch_reset)
	dbuf<uint16_t> cov_skip;
	dbuf<int32_t> cov_ex_bundle, cov_ex_l, cov_ex_r, cov_ex_cnt;
	int64_t n_cov_extra = 0;
	bool op_warp = false;                  // this batch's evidence pass runs on the warp-per-hit CIGAR walks (long CIGARs)
	bool defer_check = false;

	// pinned result mirrors, by name: owned by the context (reused by every batch it processes); the combined bundles of a group
	// pass are a batch of their own on the same context and prefix their names
	agpu_ctx *pin_ctx = NULL;
	std::string pin_tag;
	template<typename T> T *host(const std::string &name, size_t count) { return (T*)pin_ctx->pinned[pin_tag + name].ensure((count + 2) * sizeof(T)); }
};

// AGPU_DEBUG_SYNC: bit mask that puts individual stream drains back (diagnosis of ordering problems)
static int debug_sync_mask()
{
	static int m = -1;
	if(m < 0) { const char *e = getenv("AGPU_DEBUG_SYNC"); m = e ? atoi(e) : 0; }
	return m;
}
#define DEBUG_SYNC(bit) do { if(debug_sync_mask() & (bit)) TRY(stream_sync(ctx)); } while(0)

static int check_err(agpu_ctx *ctx, agpu_batch *b, const char *stage)
{
	if(b->defer_check && !(debug_sync_mask() & 2)) return AGPU_OK;        // the caller checks at its next read-back (errors are sticky counters)
	int e[ERR_WORDS];
	TRY(d2h(ctx, e, b->err.p, sizeof(e)));
	TRY(stream_sync(ctx));
	const char *names[] = {"hit order", "duplicate (pos,rpos)", "mixed strand", "rpos != pos + cigar2rlen", "junction without partial exon",
		"reserved qid", "scratch capacity", "compact input without the escape entry a sentinel announces"};
	for(int k = 0; k < 8; k++)
	{
		if(e[k] == 0) continue;
		char buf[256];
		snprintf(buf, sizeof(buf), "%s: %d violation(s) of: %s", stage, e[k], names[k]);
		ctx->last_error = buf;
		return (k == ERR_CAP) ? AGPU_ERR_CAPACITY : AGPU_ERR_INPUT;
	}
	return AGPU_OK;
}

// the combined phase sets refer to the members' coordinates: they go whenever those do (agpu_batch_phase_set), and with a new
// group pass (agpu_batch_group_bridge)
static void drop_group_phase_set(agpu_batch *b)
{
	b->gph_off.release(); b->gph_len.release(); b->gph_cnt.release(); b->gph_boff.release();
	b->gphase_built = false; b->gph_ng = 0; b->n_gphase = 0;
}

// device-wide exclusive prefix sums, one launch each (lookback.h): out[i] = sum of v[0..i), out[n] = total
static int lb_scan32(agpu_ctx *ctx, const int32_t *v, int64_t n, int mode, int64_t *out)
{
	if(mode == 0 && n <= SMALL_SCAN_MAX) { LAUNCH_B(ctx, k_small_scan_i32, 1, SMALL_SCAN_THREADS, v, n, out); return AGPU_OK; }
	LAUNCH_LB(ctx, k_lb_scan_i32, (n + 1 + LB_TILE - 1) / LB_TILE, v, n, mode, out);
	return AGPU_OK;
}
static int lb_scan64(agpu_ctx *ctx, const int64_t *v, int64_t n, int64_t *out)
{
	if(n <= SMALL_SCAN_MAX) { LAUNCH_B(ctx, k_small_scan_i64, 1, SMALL_SCAN_THREADS, v, n, out); return AGPU_OK; }
	LAUNCH_LB(ctx, k_lb_scan_i64, (n + 1 + LB_TILE - 1) / LB_TILE, v, n, out);
	return AGPU_OK;
}

// k (<= 8) int64 arrays of the same length: one launch while they fit a CTA each
static int lb_scan64_multi(agpu_ctx *ctx, int k, const int64_t *const *v, int64_t n, int64_t *const *out)
{
	if(n <= SMALL_SCAN_MAX && k <= 8)
	{
		small_scan_set s;
		memset(&s, 0, sizeof(s));
		for(int i = 0; i < k; i++) { s.in[i] = v[i]; s.out[i] = out[i]; }
		LAUNCH_B(ctx, k_small_scan_i64_multi, k, SMALL_SCAN_THREADS, s, n);
		return AGPU_OK;
	}
	for(int i = 0; i < k; i++) TRY(lb_scan64(ctx, v[i], n, out[i]));
	return AGPU_OK;
}

template<typename T> static int pull(agpu_ctx *ctx, agpu_batch *b, const std::string &name, const T *dev, size_t n, T **out)
{
	T *h = b->host<T>(name, n);
	if(!h) return AGPU_ERR_OOM;
	*out = h;
	if(n == 0 || dev == NULL) return AGPU_OK;
	ctx->d2h_result_bytes += (int64_t)(n * sizeof(T));
	return d2h(ctx, h, dev, n * sizeof(T));
}

// ------------------------------------------------------------------------------------------
extern "C" {

void agpu_default_params(agpu_params *p)
{
	p->library_type = AGPU_FR_FIRST;
	p->min_junction_support = 1;
	p->normal_junction_threshold = 10;
	p->extend_junction_threshold = 20;
	p->min_subregion_gap = 15;
	p->min_subregion_length = 15;
	p->max_reads_partition_gap = 10;
	p->bridge_end_relaxing = 10;
	p->bridge_dp_solution_size = 10;
	p->bridge_dp_stack_size = 5;
	p->insertsize_low = 80;
	p->insertsize_high = 500;
	p->max_group_size = 200;
	p->max_num_junctions_to_combine = 500;
	p->min_subregion_overlap = 1.5;
	p->min_guaranteed_edge_weight = 0.01;
	p->min_grouping_similarity = 0.10;
	p->max_grouping_similarity = 0.80;
	p->min_boundary_log_ratio = 2.0;
	p->max_group_boundary_distance = 10000;
}

int agpu_create(int device, void *stream, agpu_ctx **out)
{
	if(!out) return AGPU_ERR_ARG;
	*out = NULL;
	agpu_ctx *ctx = new (std::nothrow) agpu_ctx;
	if(!ctx) return AGPU_ERR_OOM;
	ctx->device = device;
	ctx->launches = 0;
	ctx->own_stream = false;
	ctx->stream = (cudaStream_t)stream;
	ctx->sm_count = 148;
#ifndef AGPU_EMU
	int n = 0;
	if(cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) { delete ctx; cudaGetLastError(); return AGPU_ERR_CUDA; }
	if(cudaSetDevice(device) != cudaSuccess) { delete ctx; return AGPU_ERR_CUDA; }
	cudaDeviceProp prop;
	if(cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
	if(stream == NULL)
	{
		if(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return AGPU_ERR_CUDA; }
		ctx->own_stream = true;
	}
	{
		cudaEvent_t e1, e2;
		if(cudaStreamCreateWithFlags(&ctx->side, cudaStreamNonBlocking) != cudaSuccess ||
				cudaEventCreateWithFlags(&e1, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&e2, cudaEventDisableTiming) != cudaSuccess)
		{ delete ctx; return AGPU_ERR_CUDA; }
		ctx->ev_fork = e1; ctx->ev_join = e2;
		cudaEvent_t e3;
		if(cudaEventCreateWithFlags(&e3, cudaEventDisableTiming | cudaEventBlockingSync) == cudaSuccess) ctx->ev_sync = e3;
		cudaEvent_t e4;
		if(cudaEventCreateWithFlags(&e4, cudaEventDisableTiming) == cudaSuccess) ctx->ev_stage = e4;
	}
	// keep freed blocks in the pool: the stages allocate and free stream-ordered scratch all the time
	cudaMemPool_t pool;
	if(cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess)
	{
		uint64_t thr = ~0ULL;
		cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
	}
#endif
	*out = ctx;
	return AGPU_OK;
}

void agpu_destroy(agpu_ctx *ctx)
{
	if(!ctx) return;
	AGPU_ENTER(ctx);
#ifndef AGPU_EMU
	cudaStreamSynchronize(ctx->stream);
	arena_destroy(ctx);
	lb_destroy(ctx);                      // stream-ordered frees: before the stream goes
	cudaStreamSynchronize(ctx->stream);
	if(ctx->side) { cudaStreamSynchronize(ctx->side); cudaStreamDestroy(ctx->side); }
	if(ctx->ev_fork) cudaEventDestroy((cudaEvent_t)ctx->ev_fork);
	if(ctx->ev_join) cudaEventDestroy((cudaEvent_t)ctx->ev_join);
	if(ctx->ev_sync) cudaEventDestroy((cudaEvent_t)ctx->ev_sync);
	if(ctx->ev_stage) cudaEventDestroy((cudaEvent_t)ctx->ev_stage);
	if(ctx->own_stream) cudaStreamDestroy(ctx->stream);
#endif
	pinned_free(ctx->stage_pin);
	for(auto &r : ctx->pinned) r.second.release();
#ifdef AGPU_EMU
	lb_destroy(ctx);
#endif
	delete ctx;
}

const char *agpu_last_error(agpu_ctx *ctx) { return ctx ? ctx->last_error.c_str() : "no context"; }
int agpu_sync(agpu_ctx *ctx) { if(!ctx) return AGPU_ERR_ARG; AGPU_ENTER(ctx); return stream_sync(ctx); }
int64_t agpu_launch_count(agpu_ctx *ctx) { return ctx ? ctx->launches : 0; }
int64_t agpu_sync_count(agpu_ctx *ctx) { return ctx ? ctx->syncs : 0; }
int64_t agpu_d2h_bytes(agpu_ctx *ctx) { return ctx ? ctx->d2h_result_bytes : 0; }
int agpu_pinned_match(agpu_ctx *dst, agpu_ctx *src)
{
	if(!dst || !src) return AGPU_ERR_ARG;
	if(dst == src) return AGPU_OK;
	AGPU_ENTER(dst);
	for(auto &r : src->pinned)
		if(r.second.cap > 0 && !dst->pinned[r.first].reserve_exact(r.second.cap)) return AGPU_ERR_OOM;
	return AGPU_OK;
}

// arena of the context (runtime.h): bytes held, and growth ahead of time so that a steady-state pipeline never has to take a
// new slab (a cudaMallocAsync that misses the pool synchronises the device) in the middle of its work
int64_t agpu_reserved(agpu_ctx *ctx)
{
	if(!ctx) return 0;
	int64_t tot = 0;
#ifndef AGPU_EMU
	for(size_t k = 0; k < ctx->arena.slabs.size(); k++) tot += (int64_t)ctx->arena.slabs[k].size;
#endif
	return tot;
}

int agpu_reserve(agpu_ctx *ctx, int64_t bytes)
{
	if(!ctx || bytes < 0) return AGPU_ERR_ARG;
	AGPU_ENTER(ctx);
#ifndef AGPU_EMU
	while(agpu_reserved(ctx) < bytes)
	{
		agpu_arena::slab s;
		s.size = AGPU_SLAB_BYTES; s.off = 0; s.mark = 0;
		void *base = NULL;
		if(cudaMallocAsync(&base, s.size, ctx->stream) != cudaSuccess) { cudaGetLastError(); ctx->last_error = "agpu_reserve: slab allocation failed"; return AGPU_ERR_OOM; }
		s.base = (char*)base;
		ctx->arena.slabs.push_back(s);
	}
	TRY(stream_sync(ctx));
#endif
	return AGPU_OK;
}

int agpu_upload_async(agpu_ctx *ctx, int on)
{
	if(!ctx) return AGPU_ERR_ARG;
	ctx->async_upload = on != 0;
	return AGPU_OK;
}

int agpu_blocking_sync(agpu_ctx *ctx, int on)
{
	if(!ctx) return AGPU_ERR_ARG;
#ifndef AGPU_EMU
	ctx->blocking_sync = on != 0;
#else
	(void)on;
#endif
	return AGPU_OK;
}

int agpu_profile_enable(agpu_ctx *ctx, int on) { if(!ctx) return AGPU_ERR_ARG; ctx->profiling = on != 0; return AGPU_OK; }
int agpu_profile_reset(agpu_ctx *ctx)
{
	if(!ctx) return AGPU_ERR_ARG;
	AGPU_ENTER(ctx);
	TRY(stream_sync(ctx));
	prof_collect(ctx);
	ctx->prof_acc.clear();
	return AGPU_OK;
}
int agpu_profile_read(agpu_ctx *ctx, char *buf, size_t cap)
{
	if(!ctx || !buf || cap == 0) return AGPU_ERR_ARG;
	AGPU_ENTER(ctx);
	TRY(stream_sync(ctx));
	prof_collect(ctx);
	std::string out;
	for(auto &kv : ctx->prof_acc)
	{
		char line[256];
		snprintf(line, sizeof(line), "%s\t%.6f\t%lld\n", kv.first.c_str(), kv.second.first, (long long)kv.second.second);
		out += line;
	}
	if(out.size() + 1 > cap) return AGPU_ERR_CAPACITY;
	memcpy(buf, out.c_str(), out.size() + 1);
	return AGPU_OK;
}

#define LARGE_BUNDLE_HITS 4096

// the offsets index every per-hit array: reject anything but 0 = off[0] <= ... <= off[NB] = n_hits before a kernel sees it
static int check_hit_offsets(agpu_ctx *ctx, agpu_batch *b)
{
	const std::vector<int64_t> &o = b->hit_off_host;
	bool ok = (int64_t)o.size() == (int64_t)b->nb + 1 && o[0] == 0 && o[b->nb] == b->nh;
	for(int k = 0; ok && k < b->nb; k++) ok = o[k] <= o[k + 1];
	if(!ok) { ctx->last_error = "bundle_hit_off is not a non-decreasing offset array from 0 to n_hits"; return AGPU_ERR_INPUT; }
	return AGPU_OK;
}

// average CIGAR operations per hit from which the CIGAR walks run one WARP per hit (k_hit_cigar_warp, k_cov_add_warp,
// k_hit_rpos_warp) instead of four hits per thread: at 2 operations per hit (paired-end reads) 30 of a warp's 32 lanes would idle,
// at 35 (long reads, configs[4]) the thread-per-hit walk serialises 35 dependent iterations.  AGPU_WARP_MIN_OPS=<x> overrides.
static double warp_min_ops()
{
	static double v = -1;
	if(v < 0) { const char *e = getenv("AGPU_WARP_MIN_OPS"); v = e ? atof(e) : 8.0; }
	return v;
}
static bool long_cigars(const agpu_batch *b) { return b->nh > 0 && (double)b->nc / (double)b->nh >= warp_min_ops(); }
// one warp per group of CW_WS hits, CW_WARPS warps per CTA
#define CW_GRID(ctx, n_hits) std::min<int64_t>(((n_hits) + CW_WARPS * CW_WS - 1) / (CW_WARPS * CW_WS), (int64_t)(ctx)->sm_count * 32)

// hit.rpos = pos + bam_cigar2rlen (rnacore/hit.cc:64) on the device, when the host did not send it
static int derive_rpos(agpu_ctx *ctx, agpu_batch *b)
{
	if(long_cigars(b)) LAUNCH_B(ctx, k_hit_rpos_warp, CW_GRID(ctx, b->nh), CW_WARPS * CW_WS, b->h, b->in_rpos.p);
	else LAUNCH_T(ctx, k_hit_rpos, b->nh, b->h, b->in_rpos.p);
	return AGPU_OK;
}

static int batch_common(agpu_ctx *ctx, agpu_batch *b)
{
	TRY(b->err.alloc(ctx, ERR_WORDS, true));
	std::vector<int32_t> ord(b->nb);
	for(int k = 0; k < b->nb; k++) ord[k] = k;
	const std::vector<int64_t> &ho = b->hit_off_host;
	std::stable_sort(ord.begin(), ord.end(), [&](int x, int y) { return ho[x + 1] - ho[x] > ho[y + 1] - ho[y]; });
	b->n_large = 0;
	while(b->n_large < b->nb && ho[ord[b->n_large] + 1] - ho[ord[b->n_large]] >= LARGE_BUNDLE_HITS) b->n_large++;
	// staged through the context's pinned area: asynchronous copies, no stream drain here
	const size_t need = sizeof(int32_t) * ((size_t)b->nb + 2);
#ifndef AGPU_EMU
	// the area may still feed the asynchronous copies of the previous batch of this context (agpu_upload_async, or a group
	// pass queued behind an upload): wait for those copies -- not for the stream -- before overwriting it
	if(ctx->stage_busy && ctx->ev_stage) { cudaEventSynchronize((cudaEvent_t)ctx->ev_stage); ctx->stage_busy = false; }
#endif
	if(need > ctx->stage_cap)
	{
		pinned_free(ctx->stage_pin);
		ctx->stage_cap = need * 2 + 4096;
		ctx->stage_pin = (char*)pinned_alloc(ctx->stage_cap);
		if(!ctx->stage_pin) { ctx->stage_cap = 0; return AGPU_ERR_OOM; }
	}
	int32_t *ord_pin = (int32_t*)ctx->stage_pin;
	memcpy(ord_pin, ord.data(), sizeof(int32_t) * b->nb);
	TRY(b->order.alloc(ctx, b->nb + 1));
	TRY(h2d(ctx, b->order.p, ord_pin, sizeof(int32_t) * b->nb));
#ifndef AGPU_EMU
	if(ctx->ev_stage && cudaEventRecord((cudaEvent_t)ctx->ev_stage, ctx->stream) == cudaSuccess) ctx->stage_busy = true;
	else TRY(stream_sync(ctx));
#endif
	DEBUG_SYNC(1);
	return AGPU_OK;
}

// per-bundle block-cooperative kernel over the size-binned bundle order: wide CTAs for the large bundles (few, long: on the
// side stream, next to the bulk launch), one warp for the rest
#define LAUNCH_BINNED(ctx, b, kern, ...) do { \
	bool both_ = (b)->n_large > 0 && (b)->nb > (b)->n_large; \
	if(both_) { side_fork(ctx); LAUNCH_B_SIDE(ctx, kern, (b)->n_large, 256, (b)->order.p, (b)->n_large, __VA_ARGS__); } \
	else if((b)->n_large > 0) LAUNCH_B(ctx, kern, (b)->n_large, 256, (b)->order.p, (b)->n_large, __VA_ARGS__); \
	if((b)->nb > (b)->n_large) LAUNCH_B(ctx, kern, (b)->nb - (b)->n_large, 32, (b)->order.p + (b)->n_large, (b)->nb - (b)->n_large, __VA_ARGS__); \
	if(both_) side_join(ctx); } while(0)


int agpu_batch_upload(agpu_ctx *ctx, const agpu_batch_in *in, agpu_batch **out)
{
	if(!ctx || !in || !out || in->n_bundles < 0 || in->n_hits < 0) return AGPU_ERR_ARG;
	AGPU_ENTER(ctx);
	*out = NULL;
	agpu_batch *b = new (std::nothrow) agpu_batch;
	if(!b) return AGPU_ERR_OOM;
	b->nb = in->n_bundles; b->nh = in->n_hits; b->nc = in->n_cigar;
	b->pin_ctx = ctx;
	b->owns_input = true;
	b->hit_off_host.assign(in->bundle_hit_off, in->bundle_hit_off + b->nb + 1);
	b->tid_host.assign(in->bundle_tid, in->bundle_tid + b->nb);
	if(in->bundle_sample) b->sample_host.assign(in->bundle_sample, in->bundle_sample + b->nb);
	int rc = check_hit_offsets(ctx, b);
	if(rc != AGPU_OK) { delete b; return rc; }
	// the uploaded inputs live at the bottom of the context's arena too (below the mark a reset rewinds to): a pipeline in
	// steady state then makes no allocator call at all
	if(ctx->arena_owner == NULL) { ctx->arena_owner = b; ctx->arena.rewind(); }
	arena_scope input_scope(ctx, b);
#define UP(buf, src, count) do { if(rc == AGPU_OK) rc = b->buf.alloc(ctx, (size_t)(count) + 1); if(rc == AGPU_OK) rc = h2d(ctx, b->buf.p, src, sizeof(*(src)) * (size_t)(count)); } while(0)
	UP(in_hit_off, in->bundle_hit_off, b->nb + 1);
	UP(in_pos, in->pos, b->nh); UP(in_mpos, in->mpos, b->nh); UP(in_isize, in->isize, b->nh);
	UP(in_xs, in->xs, b->nh); UP(in_qid, in->qid, b->nh);
	// flag[] is not read by any kernel and stays on the host; rpos[] and strand[] are optional (see agpu_batch_in)
	if(in->rpos) UP(in_rpos, in->rpos, b->nh);
	if(in->strand) UP(in_strand, in->strand, b->nh);
	else if(in->bundle_strand) UP(in_bstrand, in->bundle_strand, b->nb);
	else rc = rc == AGPU_OK ? AGPU_ERR_ARG : rc;
	UP(in_cigar_off, in->cigar_off, b->nh + 1); UP(in_cigar, in->cigar, b->nc);
#undef UP
	if(rc == AGPU_OK) rc = batch_common(ctx, b);
	if(rc != AGPU_OK) { agpu_batch_free(ctx, b); return rc; }
	b->h.n_hits = b->nh; b->h.n_bundles = b->nb;
	b->h.bundle_hit_off = b->in_hit_off.p;
	b->h.pos = b->in_pos.p; b->h.rpos = b->in_rpos.p; b->h.mpos = b->in_mpos.p; b->h.isize = b->in_isize.p;
	b->h.flag = NULL; b->h.strand = b->in_strand.p; b->h.bundle_strand = b->in_bstrand.p; b->h.xs = b->in_xs.p; b->h.qid = (const u64*)b->in_qid.p;
	b->h.cigar_off = b->in_cigar_off.p; b->h.cigar = b->in_cigar.p;
	if(!in->rpos)
	{
		// hit.rpos = pos + bam_cigar2rlen (rnacore/hit.cc:64), derived on the device
		if(b->in_rpos.alloc(ctx, (size_t)b->nh + 1) != AGPU_OK) { agpu_batch_free(ctx, b); return AGPU_ERR_OOM; }
		b->h.rpos = b->in_rpos.p;
		if(derive_rpos(ctx, b) != AGPU_OK) { agpu_batch_free(ctx, b); return AGPU_ERR_CUDA; }
	}
	if(ctx->arena_owner == b) ctx->arena.set_mark();
	// the caller's buffers (and the context's staging area) are free again when this returns -- unless the context uploads
	// asynchronously (agpu_upload_async): then they are when the batch's first stage call returns
	if(!ctx->async_upload && stream_sync(ctx) != AGPU_OK) { agpu_batch_free(ctx, b); return AGPU_ERR_CUDA; }
	*out = b;
	return AGPU_OK;
}

int agpu_batch_adopt(agpu_ctx *ctx, const agpu_batch_in *in, agpu_batch **out)
{
	if(!ctx || !in || !out || in->n_bundles < 0 || in->n_hits < 0) return AGPU_ERR_ARG;
	AGPU_ENTER(ctx);
	*out = NULL;
	agpu_batch *b = new (std::nothrow) agpu_batch;
	if(!b) return AGPU_ERR_OOM;
	b->nb = in->n_bundles; b->nh = in->n_hits; b->nc = in->n_cigar;
	b->pin_ctx = ctx;
	b->owns_input = false;
	b->hit_off_host.resize(b->nb + 1);
	b->tid_host.resize(b->nb);
	if(ctx->arena_owner == NULL) { ctx->arena_owner = b; ctx->arena.rewind(); }
	arena_scope input_scope(ctx, b);
	int rc = d2h(ctx, b->hit_off_host.data(), in->bundle_hit_off, sizeof(int64_t) * (b->nb + 1));
	if(rc == AGPU_OK) rc = d2h(ctx, b->tid_host.data(), in->bundle_tid, sizeof(int32_t) * b->nb);
	if(rc == AGPU_OK && in->bundle_sample) { b->sample_host.resize(b->nb); rc = d2h(ctx, b->sample_host.data(), in->bundle_sample, sizeof(int32_t) * b->nb); }
	if(rc == AGPU_OK) rc = stream_sync(ctx);
	if(rc == AGPU_OK) rc = check_hit_offsets(ctx, b);
	if(rc == AGPU_OK) rc = batch_common(ctx, b);
	if(rc != AGPU_OK) { agpu_batch_free(ctx, b); return rc; }
	b->h.n_hits = b->nh; b->h.n_bundles = b->nb;
	b->h.bundle_hit_off = in->bundle_hit_off;
	b->h.pos = in->pos; b->h.rpos = in->rpos; b->h.mpos = in->mpos; b->h.isize = in->isize;
	b->h.flag = in->flag; b->h.strand = in->strand; b->h.bundle_strand = in->bundle_strand; b->h.xs = in->xs; b->h.qid = (const u64*)in->qid;
	b->h.cigar_off = in->cigar_off; b->h.cigar = in->cigar;
	if(!in->strand && !in->bundle_strand) { agpu_batch_free(ctx, b); return AGPU_ERR_ARG; }
	if(!in->rpos)
	{
		if(b->in_rpos.alloc(ctx, (size_t)b->nh + 1) != AGPU_OK) { agpu_batch_free(ctx, b); return AGPU_ERR_OOM; }
		b->h.rpos = b->in_rpos.p;
		if(derive_rpos(ctx, b) != AGPU_OK) { agpu_batch_free(ctx, b); return AGPU_ERR_CUDA; }
	}
	if(ctx->arena_owner == b) ctx->arena.set_mark();
	if(stream_sync(ctx) != AGPU_OK) { agpu_batch_free(ctx, b); return AGPU_ERR_CUDA; }      // frees the context's staging area
	*out = b;
	return AGPU_OK;
}

static void release_derived(agpu_ctx *ctx, agpu_batch *b)
{
	if(b->cb) agpu_batch_free(ctx, b->cb);
	static_cast<batch_derived&>(*b) = batch_derived();
}

void agpu_batch_free(agpu_ctx *ctx, agpu_batch *b)
{
	if(!ctx || !b) return;
	AGPU_ENTER(ctx);
	release_derived(ctx, b);
	stream_sync(ctx);
	if(ctx->arena_owner == b) { ctx->arena.rewind(); ctx->arena_owner = NULL; }
	delete b;                             // the inputs: frees inside the arena's slabs are no-ops
}

int agpu_batch_reset(agpu_ctx *ctx, agpu_batch *b)
{
	if(!ctx || !b) return AGPU_ERR_ARG;
	AGPU_ENTER(ctx);
	release_derived(ctx, b);
	if(ctx->arena_owner == b) ctx->arena.rewind_to_mark();
	TRY(b->err.fill(ctx, 0));
	return AGPU_OK;
}

// ---- chain set construction shared by hcst (elements = hits) and fcst (elements = fragments)
// Table regions: a power of two >= 2 x the elements that will be inserted.  `d_count` (device, per bundle) gives that number
// when only some elements carry a chain (hcst: the spliced hits); otherwise every element of the bundle counts.
// table regions: a power of two >= 2 x the bundle's count.  With per-bundle counts (d_count: the spliced hits, far fewer than the
// elements) the total is read back; without, the regions are sized from the element offsets on the device and the table is
// allocated by its bound (a power of two below 4 x count), with no read-back at all
static int chainset_build(agpu_ctx *ctx, agpu_batch *b, chainset_state &cs, int64_t n_elem, const int64_t *d_elem_off, const int32_t *d_count = NULL)
{
	int nb = b->nb;
	cs.n_elem = n_elem;
	cs.d_elem_off = d_elem_off;
	TRY(cs.reg_off.alloc(ctx, nb + 2));
	if(d_count)
	{
		dbuf<int64_t> sz;
		TRY(sz.alloc(ctx, nb + 1));
		LAUNCH_T(ctx, k_table_sizes, nb, nb, d_count, sz.p);
		TRY(lb_scan64(ctx, sz.p, nb, cs.reg_off.p));
		TRY(d2h(ctx, &cs.n_slots, cs.reg_off.p + nb, sizeof(int64_t)));
		TRY(stream_sync(ctx));
	}
	else
	{
		dbuf<int64_t> sz;
		TRY(sz.alloc(ctx, nb + 1));
		LAUNCH_T(ctx, k_table_sizes_off, nb, nb, d_elem_off, sz.p);
		TRY(lb_scan64(ctx, sz.p, nb, cs.reg_off.p));
		cs.n_slots = 4 * n_elem + 2 * (int64_t)nb;
		DEBUG_SYNC(16);
	}
	TRY(cs.slot_word.alloc(ctx, cs.n_slots, true));
	TRY(cs.slot_first.alloc(ctx, cs.n_slots)); TRY(cs.slot_first.fill(ctx, 0x7f));
	TRY(cs.slot_cnt.alloc(ctx, cs.n_slots * 3, true));
	TRY(cs.slot_chain.alloc(ctx, cs.n_slots));
	TRY(cs.elem_slot.alloc(ctx, n_elem));
	TRY(cs.n_chains.alloc(ctx, nb, true)); TRY(cs.n_splices.alloc(ctx, nb, true));
	TRY(cs.c_rep.alloc(ctx, n_elem)); TRY(cs.c_cnt.alloc(ctx, n_elem * 3)); TRY(cs.c_grp.alloc(ctx, n_elem)); TRY(cs.c_slot.alloc(ctx, n_elem));
	TRY(cs.handle_chain.alloc(ctx, n_elem));
	TRY(cs.key_scratch.alloc(ctx, n_elem));
	return AGPU_OK;
}

static int chainset_finish(agpu_ctx *ctx, agpu_batch *b, chainset_state &cs, int64_t n_val)
{
	LAUNCH_BINNED(ctx, b, k_chain_order, cs.d_elem_off, cs.elem_slot.p, cs.slot_first.p, cs.slot_cnt.p, cs.voff32, cs.voff64, cs.val,
			cs.key_scratch.p, cs.slot_chain.p, cs.n_chains.p, cs.c_rep.p, cs.c_cnt.p, cs.c_grp.p, cs.c_slot.p);
	TRY(cs.key_scratch2.alloc(ctx, 2 * n_val + 2));
	TRY(cs.splices_scratch.alloc(ctx, n_val + 1));
	LAUNCH_BINNED(ctx, b, k_chain_splices, cs.d_elem_off, cs.val_base.p, cs.n_chains.p, cs.c_rep.p, cs.c_cnt.p,
			cs.elem_len, cs.voff32, cs.voff64, cs.val, cs.key_scratch2.p, cs.n_splices.p, cs.splices_scratch.p);
	LAUNCH_T(ctx, k_handle_chain, cs.n_elem, cs.n_elem, cs.elem_slot.p, cs.slot_chain.p, cs.handle_chain.p);
	cs.built = true;
	return AGPU_OK;
}

// border bitmap + hits (+ the stretches of update_bridges) -> ranked borders, differences, coverage, segments.  One stream drain:
// the border count, which sizes the per-border arrays.  The segment count stays on the device (cov_tot[1]) and is read back
// with the next read-back that needs it (seg_count).
static int coverage_scan(agpu_ctx *ctx, agpu_batch *b)
{
	const int nb = b->nb;
	TRY(b->seg_off.alloc(ctx, nb + 2, true));
	b->n_seg = 0; b->n_bord = 0; b->n_seg_on_dev = false;
	const int64_t nw = b->ltot / 32;
	TRY(b->cov_tot.alloc(ctx, 4, true));
	if(nw > 0)
	{
		// rank the borders: one look-back pass over the bitmap words
		TRY(b->wrank.alloc(ctx, nw + 2));
		LAUNCH_LB(ctx, k_lb_bord_rank, (nw + 1 + LB_TILE - 1) / LB_TILE, b->border.p, nw, b->wrank.p, b->cov_tot.p);
		TRY(d2h(ctx, &b->n_bord, b->cov_tot.p, sizeof(int64_t)));
		TRY(stream_sync(ctx));
	}
	const int64_t n = b->n_bord;
	TRY(b->seg_l.alloc(ctx, n + 1)); TRY(b->seg_r.alloc(ctx, n + 1)); TRY(b->seg_c.alloc(ctx, n + 1));
	if(n > 0)
	{
		TRY(b->diffc.alloc(ctx, n + 1, true)); TRY(b->posc.alloc(ctx, n + 1));
		const int64_t n_tiles = (n + 1 + LB_TILE - 1) / LB_TILE;      // tiles of k_lb_cov_segments
		dbuf<int32_t> tile_b0;
		TRY(b->bord_off.alloc(ctx, nb + 2)); TRY(tile_b0.alloc(ctx, n_tiles + 1));
		LAUNCH_T(ctx, k_bord_off, nb + 1, nb, b->cov_base.p, b->wrank.p, b->bord_off.p, n_tiles, tile_b0.p);
		LAUNCH_B(ctx, k_bord_positions, (nw + LB_TILE - 1) / LB_TILE, 256, nw, b->border.p, b->wrank.p, nb, b->cov_base.p, b->b_lpos.p, b->posc.p);
		if(b->op_warp) LAUNCH_B(ctx, k_cov_add_warp, CW_GRID(ctx, b->nh), CW_WARPS * CW_WS, b->h, b->hit_bundle.p, b->b_lpos.p, b->cov_base.p, b->border.p, b->wrank.p, b->diffc.p, b->cov_skip.p);
		else LAUNCH_T(ctx, k_cov_add, HQ_THREADS(b->nh), b->h, b->hit_bundle.p, b->b_lpos.p, b->cov_base.p, b->border.p, b->wrank.p, b->diffc.p, b->cov_skip.p);
		LAUNCH_T(ctx, k_cov_add_extra, b->n_extra, b->n_extra, b->ex_s.p, b->ex_e.p, b->border.p, b->wrank.p, b->diffc.p);
		LAUNCH_T(ctx, k_cov_add_points, b->n_pts, b->n_pts, b->pt_g.p, b->pt_d.p, b->border.p, b->wrank.p, b->diffc.p);
		// coverage = prefix sum of the differences; segments = borders with positive coverage; prefix sums of len * cov:
		// one launch, three chained look-backs.  Then the run structure.  Both are sized by the border count, an upper bound of the
		// segment count
		dbuf<uint8_t> s_head;
		TRY(s_head.alloc(ctx, n + 1)); TRY(b->seg_psum.alloc(ctx, n + 2)); TRY(b->seg_nhead.alloc(ctx, n + 2));
		LAUNCH_LB(ctx, k_lb_cov_segments, n_tiles, b->diffc.p, b->posc.p, n, nb, b->bord_off.p, tile_b0.p,
				b->seg_l.p, b->seg_r.p, b->seg_c.p, b->seg_off.p, s_head.p, b->seg_psum.p, b->cov_tot.p + 1);
		LAUNCH_B(ctx, k_seg_nhead, (n + LB_TILE - 1) / LB_TILE, LB_THREADS, n, s_head.p, b->cov_tot.p + 1, b->seg_nhead.p);
		b->n_seg_on_dev = true;
	}
	else TRY(b->seg_psum.alloc(ctx, 2, true));
	b->cov_dirty = false;
	return AGPU_OK;
}

// queue the copy of the segment count coverage_scan left on the device; b->n_seg holds it after the caller's next stream drain
static int seg_count(agpu_ctx *ctx, agpu_batch *b)
{
	if(!b->n_seg_on_dev) return AGPU_OK;
	TRY(d2h(ctx, &b->n_seg, b->cov_tot.p + 1, sizeof(int64_t)));
	b->n_seg_on_dev = false;
	return AGPU_OK;
}

int agpu_batch_evidence(agpu_ctx *ctx, agpu_batch *b, const agpu_params *p)
{
	if(!ctx || !b || !p) return AGPU_ERR_ARG;
	AGPU_ENTER(ctx);
	AGPU_BATCH_SCOPE(ctx, b);
	if(b->evidence) return AGPU_OK;
	int nb = b->nb;
	int64_t nh = b->nh, nc = b->nc;
	TRY(b->b_lpos.alloc(ctx, nb + 1)); TRY(b->b_rpos.alloc(ctx, nb + 1)); TRY(b->b_covhi.alloc(ctx, nb + 1));
	TRY(b->b_strand.alloc(ctx, nb + 1)); TRY(b->b_span.alloc(ctx, nb + 1)); TRY(b->cov_base.alloc(ctx, nb + 2));
	TRY(b->hit_bundle.alloc(ctx, nh + 1));
	{
		dbuf<int32_t> npq, tile_bundle;
		const int64_t n_tiles = (nh + HB_TILE - 1) / HB_TILE;
		TRY(npq.alloc(ctx, 2 * (size_t)nb + 2)); TRY(tile_bundle.alloc(ctx, (size_t)n_tiles + 2));
		LAUNCH_T(ctx, k_bundle_init, nb, nb, b->b_lpos.p, b->b_rpos.p, b->b_covhi.p, npq.p);
		LAUNCH_T(ctx, k_tile_bundle, n_tiles + 1, b->h, n_tiles, tile_bundle.p);
		LAUNCH_T(ctx, k_hit_bounds, nh, b->h, tile_bundle.p, b->b_lpos.p, b->b_rpos.p, b->b_covhi.p, npq.p, b->hit_bundle.p, b->err.p);
		LAUNCH_T(ctx, k_bundle_finish, nb, b->h, p->library_type, b->b_lpos.p, b->b_covhi.p, npq.p, b->b_strand.p, b->b_span.p);
	}
	TRY(lb_scan64(ctx, b->b_span.p, nb, b->cov_base.p));
	b->ltot = 0;
	TRY(d2h(ctx, &b->ltot, b->cov_base.p + nb, sizeof(int64_t)));
	TRY(stream_sync(ctx));
	if(b->ltot >= ((int64_t)1 << 32) - 64) { ctx->last_error = "batch spans 2^32 or more window positions: split it"; return AGPU_ERR_CAPACITY; }
	TRY(b->border.alloc(ctx, b->ltot / 32 + 8, true));
	TRY(b->spl.alloc(ctx, nc + 1)); TRY(b->hit_nspl.alloc(ctx, nh + 1, true));
	dbuf<int32_t> n_spliced;
	TRY(n_spliced.alloc(ctx, nb + 1, true));
	// CIGAR walk: four hits per thread (k_hit_cigar here, k_cov_add after the borders are ranked), or one warp per hit for batches
	// of long CIGARs (warp_min_ops)
	b->op_warp = long_cigars(b);
	if(b->op_warp) LAUNCH_B(ctx, k_hit_cigar_warp, CW_GRID(ctx, nh), CW_WARPS * CW_WS, b->h, b->b_lpos.p, b->cov_base.p, b->border.p, b->spl.p, b->hit_nspl.p, b->hit_bundle.p, n_spliced.p, b->err.p, b->cov_skip.p);
	else LAUNCH_T(ctx, k_hit_cigar, HQ_THREADS(nh), b->h, b->b_lpos.p, b->cov_base.p, b->border.p, b->spl.p, b->hit_nspl.p, b->hit_bundle.p, n_spliced.p, b->err.p, b->cov_skip.p);
	if(b->n_cov_extra > 0)
	{
		// foreign intervals of the insert-size preview (agpu_batch_coverage_edit): border bits now, weights with the ranked borders
		b->n_pts = 2 * b->n_cov_extra;
		TRY(b->pt_g.alloc(ctx, b->n_pts + 1)); TRY(b->pt_d.alloc(ctx, b->n_pts + 1));
		LAUNCH_T(ctx, k_extra_intervals, b->n_cov_extra, b->n_cov_extra, b->cov_ex_bundle.p, b->cov_ex_l.p, b->cov_ex_r.p, b->cov_ex_cnt.p, b->b_lpos.p,
				b->b_covhi.p, b->cov_base.p, b->border.p, b->pt_g.p, b->pt_d.p);
	}
	// hcst
	chainset_state &cs = b->hcst;
	cs.val = b->spl.p; cs.voff32 = b->h.cigar_off; cs.voff64 = NULL; cs.elem_len = b->hit_nspl.p;
	TRY(chainset_build(ctx, b, cs, nh, b->h.bundle_hit_off, n_spliced.p));
	n_spliced.release();
	LAUNCH_T(ctx, k_hcst_insert, nh, b->h, b->hit_nspl.p, b->hit_bundle.p, b->spl.p, cs.reg_off.p, cs.slot_word.p,
			cs.slot_first.p, cs.slot_cnt.p, cs.elem_slot.p, b->err.p);
	TRY(cs.val_base.alloc(ctx, nb + 1));
	LAUNCH_T(ctx, k_gather_off, nb + 1, nb + 1, b->h.bundle_hit_off, b->h.cigar_off, cs.val_base.p);
	TRY(chainset_finish(ctx, b, cs, nc));
	TRY(coverage_scan(ctx, b));
	b->evidence = true;
	return check_err(ctx, b, "agpu_batch_evidence");
}

int agpu_batch_graph(agpu_ctx *ctx, agpu_batch *b, const agpu_params *p)
{
	if(!ctx || !b || !p) return AGPU_ERR_ARG;
	AGPU_ENTER(ctx);
	AGPU_BATCH_SCOPE(ctx, b);
	if(!b->evidence) return AGPU_ERR_ARG;
	if(b->cov_dirty) TRY(coverage_scan(ctx, b));
	graph_state &gs = b->gr;
	gs = graph_state();
	int nb = b->nb;
	graph_in in;
	in.n = nb; in.lpos = b->b_lpos.p; in.rpos = b->b_rpos.p; in.strand = b->b_strand.p;
	in.hc = b->hcst.view(); in.fc = b->fcst.view();
	in.seg_off = b->seg_off.p; in.seg_l = b->seg_l.p; in.seg_r = b->seg_r.p; in.seg_c = b->seg_c.p;
	in.seg_nhead = b->seg_nhead.p; in.seg_psum = b->seg_psum.p;
	for(int k = 0; k < 5; k++) { TRY(gs.ub[k].alloc(ctx, nb + 1)); TRY(gs.off[k].alloc(ctx, nb + 2)); }
	LAUNCH_B(ctx, k_graph_bounds, nb, 128, in, gs.ub[0].p, gs.ub[1].p, gs.ub[2].p, gs.ub[3].p, gs.ub[4].p);
	{
		const int64_t *in5[5]; int64_t *out5[5];
		for(int k = 0; k < 5; k++) { in5[k] = gs.ub[k].p; out5[k] = gs.off[k].p; }
		TRY(lb_scan64_multi(ctx, 5, in5, nb, out5));
		for(int k = 0; k < 5; k++) TRY(d2h(ctx, &gs.tot[k], gs.off[k].p + nb, sizeof(int64_t)));
	}
	TRY(stream_sync(ctx));
	int64_t J = gs.tot[0], P = gs.tot[1], E = gs.tot[2];
	int64_t V = P + 2 * (int64_t)nb, VO = P + 3 * (int64_t)nb;
	TRY(gs.iarena.alloc(ctx, gs.tot[3] + 16)); TRY(gs.karena.alloc(ctx, gs.tot[4] + 16));
	TRY(gs.n_junc.alloc(ctx, nb + 1, true)); TRY(gs.n_pex.alloc(ctx, nb + 1, true)); TRY(gs.n_edge.alloc(ctx, nb + 1, true));
	for(int k = 0; k < 9; k++) TRY(gs.j[k].alloc(ctx, J + 1));
	for(int k = 0; k < 6; k++) { TRY(gs.p_i[k].alloc(ctx, P + 1)); TRY(gs.v_i[k].alloc(ctx, V + 1)); }
	for(int k = 0; k < 3; k++) { TRY(gs.p_d[k].alloc(ctx, P + 1)); TRY(gs.v_d[k].alloc(ctx, V + 1)); TRY(gs.e_i[k].alloc(ctx, E + 1)); }
	TRY(gs.e_w.alloc(ctx, E + 1));
	TRY(gs.in_off.alloc(ctx, VO + 1)); TRY(gs.in_src.alloc(ctx, E + 1)); TRY(gs.in_eid.alloc(ctx, E + 1));
	TRY(gs.out_off.alloc(ctx, VO + 1)); TRY(gs.out_dst.alloc(ctx, E + 1)); TRY(gs.out_eid.alloc(ctx, E + 1));
	graph_params gp;
	gp.min_junction_support = p->min_junction_support;
	gp.min_subregion_gap = p->min_subregion_gap; gp.min_subregion_length = p->min_subregion_length;
	gp.min_subregion_overlap = p->min_subregion_overlap; gp.min_guaranteed_edge_weight = p->min_guaranteed_edge_weight;
	LAUNCH_BINNED(ctx, b, k_graph_build, in, gs.dev(b->err.p), gp);
	gs.built = true;
	return check_err(ctx, b, "agpu_batch_graph");
}

#include "abi_stages.inc"
#include "abi_fetch.inc"
#include "abi_group.inc"
#include "abi_phase.inc"
#include "abi_revise.inc"
#include "abi_support.inc"
#include "abi_preview.inc"
#include "abi_packed.inc"
#include "abi_regroup.inc"

}
