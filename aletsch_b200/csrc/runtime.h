// Host-side runtime of libaletsch_gpu.so: context, stream-ordered device buffers, launch macros.
#ifndef ALETSCH_B200_CSRC_RUNTIME_H
#define ALETSCH_B200_CSRC_RUNTIME_H

#include "dev.h"
#include "lookback.h"
#include "../../include/aletsch_gpu.h"

#include <map>
#include <string>
#include <vector>

struct agpu_batch;
struct agpu_prof_rec { const char *name; void *e0, *e1; };

// pinned host array (results): grown on demand, kept by the context
struct agpu_pinbuf
{
	char *p = NULL;
	size_t cap = 0;
	char *ensure(size_t bytes);
	bool reserve_exact(size_t bytes);     // grow to exactly `bytes` if smaller (contents are not kept)
	void release();
};

// Bump arena for the derived state of ONE batch per context: a few large slabs taken from the stream-ordered pool once and
// kept for the context's lifetime.  The stages allocate ~150 arrays per step; bumping a pointer instead of going through
// cudaMallocAsync / cudaFreeAsync removes that API time and, with several contexts working side by side (pipeline.py), the
// cross-stream reuse dependencies of the shared pool.  Individual frees are no-ops; the arena rewinds at batch reset / free.
struct agpu_arena
{
	// First fit over all slabs: a request goes to the first slab with room for it, so the tail a large request could not use is
	// still filled by the smaller ones that follow, and a batch whose big arrays are a little larger than the previous batch's
	// does not strand the slabs sized for those (a strictly forward-moving cursor did: the pool's contexts kept adding slabs
	// until the device was full).
	struct slab { char *base; size_t size; size_t off; size_t mark; };
	std::vector<slab> slabs;
	bool contains(const void *p) const
	{
		for(size_t k = 0; k < slabs.size(); k++) if((const char*)p >= slabs[k].base && (const char*)p < slabs[k].base + slabs[k].size) return true;
		return false;
	}
	// end of the batch's uploaded inputs: a reset rewinds to here, a free to 0
	void set_mark() { for(size_t k = 0; k < slabs.size(); k++) slabs[k].mark = slabs[k].off; }
	void rewind_to_mark() { for(size_t k = 0; k < slabs.size(); k++) slabs[k].off = slabs[k].mark; }
	void rewind() { for(size_t k = 0; k < slabs.size(); k++) slabs[k].off = slabs[k].mark = 0; }
};

struct agpu_ctx
{
	int device;
	cudaStream_t stream;
	bool own_stream;
	int64_t launches;
	std::string last_error;
	int sm_count;
	agpu_arena arena;
	agpu_batch *arena_owner = NULL;     // the batch whose stages allocate from the arena
	bool arena_on = false;              // set while a stage of the owner runs
	// side stream: runs the few-but-long launches of a size-binned kernel pair next to the bulk launch on `stream`
	cudaStream_t side = NULL;
	void *ev_fork = NULL, *ev_join = NULL;
	// host waits: spin on the stream (lowest latency) or sleep on an event created with cudaEventBlockingSync (many host threads
	// per core, e.g. eight ranks with a stream pool each on one box)
	bool blocking_sync = false;
	void *ev_sync = NULL;
	// small pinned staging area for the per-bundle tables an upload derives on the host (grown on demand, reused by every batch
	// of the context).  The copies out of it are asynchronous: ev_stage is recorded behind them and the next user of the area
	// waits for that event first, so a second upload / group pass on the same context cannot overwrite tables still in flight.
	char *stage_pin = NULL;
	size_t stage_cap = 0;
	void *ev_stage = NULL;
	bool stage_busy = false;
	// decoupled look-back scans (lookback.h): status words, ticket counter, launch epoch, tickets consumed so far
	unsigned long long *lb_status = NULL, *lb_ticket = NULL;
	int64_t lb_stride = 0;
	unsigned long long lb_tickets = 0;
	unsigned lb_epoch = 0;
	// pinned result mirrors of the fetches, by name (see agpu_batch::host)
	std::map<std::string, agpu_pinbuf> pinned;
	int64_t syncs = 0;
	int64_t d2h_result_bytes = 0;       // bytes the result fetches copied device -> host (agpu_d2h_bytes)
	// agpu_upload_async: the uploads of this context return as soon as their copies and decode kernels are queued
	bool async_upload = false;
	// optional per-kernel timing (CUDA events around every launch on the ctx stream)
	bool profiling = false;
	std::vector<agpu_prof_rec> prof;
	std::vector<void*> free_events;
	std::map<std::string, std::pair<double, int64_t> > prof_acc;    // name -> (ms, launches)
};

namespace agpu {

#ifndef AGPU_EMU
#define CUDA_TRY(ctx, call) do { cudaError_t e_ = (call); if(e_ != cudaSuccess) { (ctx)->last_error = std::string(#call) + ": " + cudaGetErrorString(e_); return AGPU_ERR_CUDA; } } while(0)

inline void prof_begin(agpu_ctx *ctx, const char *name, cudaStream_t st = NULL)
{
	if(!ctx->profiling) return;
	if(st == NULL) st = ctx->stream;
	agpu_prof_rec r;
	r.name = name;
	cudaEvent_t e[2];
	for(int k = 0; k < 2; k++)
	{
		if(!ctx->free_events.empty()) { e[k] = (cudaEvent_t)ctx->free_events.back(); ctx->free_events.pop_back(); }
		else cudaEventCreate(&e[k]);
	}
	r.e0 = e[0]; r.e1 = e[1];
	cudaEventRecord(e[0], st);
	ctx->prof.push_back(r);
}
inline void prof_end(agpu_ctx *ctx, cudaStream_t st = NULL)
{
	if(!ctx->profiling) return;
	cudaEventRecord((cudaEvent_t)ctx->prof.back().e1, st ? st : ctx->stream);
}
// side stream joins in after everything queued on the main stream so far / main stream waits for the side stream
inline void side_fork(agpu_ctx *ctx) { cudaEventRecord((cudaEvent_t)ctx->ev_fork, ctx->stream); cudaStreamWaitEvent(ctx->side, (cudaEvent_t)ctx->ev_fork, 0); }
inline void side_join(agpu_ctx *ctx) { cudaEventRecord((cudaEvent_t)ctx->ev_join, ctx->side); cudaStreamWaitEvent(ctx->stream, (cudaEvent_t)ctx->ev_join, 0); }
// block-cooperative kernel on the side stream (between side_fork and side_join)
#define LAUNCH_B_SIDE(ctx, kern, nblocks, nthreads, ...) do { int64_t n_ = (int64_t)(nblocks); if(n_ > 0) { unsigned g_ = (unsigned)(n_ > 1048576 ? 1048576 : n_); \
	prof_begin(ctx, #kern "(side)", (ctx)->side); kern<<<g_, (nthreads), 0, (ctx)->side>>>(__VA_ARGS__); prof_end(ctx, (ctx)->side); (ctx)->launches++; } } while(0)
// fold finished records into the per-kernel accumulators (call after a stream synchronisation)
inline void prof_collect(agpu_ctx *ctx)
{
	for(size_t k = 0; k < ctx->prof.size(); k++)
	{
		float ms = 0;
		agpu_prof_rec &r = ctx->prof[k];
		if(cudaEventElapsedTime(&ms, (cudaEvent_t)r.e0, (cudaEvent_t)r.e1) == cudaSuccess)
		{
			std::pair<double, int64_t> &a = ctx->prof_acc[r.name];
			a.first += ms; a.second += 1;
		}
		else cudaGetLastError();
		ctx->free_events.push_back(r.e0); ctx->free_events.push_back(r.e1);
	}
	ctx->prof.clear();
}

// entry points may be called from any host thread: the CUDA current device is per thread
#define AGPU_ENTER(ctx) do { cudaSetDevice((ctx)->device); } while(0)

// per-thread kernel: grid covers n items
#define LAUNCH_T(ctx, kern, n, ...) do { int64_t n_ = (int64_t)(n); if(n_ > 0) { unsigned g_ = (unsigned)((n_ + 255) / 256); \
	prof_begin(ctx, #kern); kern<<<g_, 256, 0, (ctx)->stream>>>(__VA_ARGS__); prof_end(ctx); (ctx)->launches++; } } while(0)
// block-cooperative kernel: one CTA per work item (the kernel loops if the grid is smaller)
#define LAUNCH_B(ctx, kern, nblocks, nthreads, ...) do { int64_t n_ = (int64_t)(nblocks); if(n_ > 0) { unsigned g_ = (unsigned)(n_ > 1048576 ? 1048576 : n_); \
	prof_begin(ctx, #kern); kern<<<g_, (nthreads), 0, (ctx)->stream>>>(__VA_ARGS__); prof_end(ctx); (ctx)->launches++; } } while(0)

#define AGPU_SLAB_BYTES ((size_t)1 << 30)
inline void *arena_alloc(agpu_ctx *ctx, size_t bytes)
{
	agpu_arena &a = ctx->arena;
	bytes = (bytes + 255) & ~(size_t)255;
	for(size_t k = 0; k < a.slabs.size(); k++)
		if(a.slabs[k].off + bytes <= a.slabs[k].size) { void *p = a.slabs[k].base + a.slabs[k].off; a.slabs[k].off += bytes; return p; }
	agpu_arena::slab s;
	// an oversize request gets a slab of its own with 1/8 of headroom, rounded to 256 MB: the next batch's array of the same kind
	// is rarely exactly as large
	s.size = AGPU_SLAB_BYTES;
	if(bytes > AGPU_SLAB_BYTES) s.size = (bytes + bytes / 8 + ((size_t)1 << 28) - 1) & ~(((size_t)1 << 28) - 1);
	s.off = 0; s.mark = 0;
	void *base = NULL;
	if(cudaMallocAsync(&base, s.size, ctx->stream) != cudaSuccess)
	{
		cudaGetLastError();
		size_t fr = 0, tot = 0, held = 0;
		cudaMemGetInfo(&fr, &tot);
		for(size_t k = 0; k < a.slabs.size(); k++) held += a.slabs[k].size;
		char buf[256];
		snprintf(buf, sizeof(buf), "arena slab allocation of %zu MB failed: context holds %zu slabs / %zu MB, device free %zu MB of %zu MB",
				s.size >> 20, a.slabs.size(), held >> 20, fr >> 20, tot >> 20);
		ctx->last_error = buf;
		return NULL;
	}
	s.base = (char*)base;
	s.off = bytes;
	a.slabs.push_back(s);
	return s.base;
}
inline int dev_alloc_bytes(agpu_ctx *ctx, void **p, size_t bytes, bool zero)
{
	*p = NULL;
	if(bytes == 0) bytes = 16;
	cudaError_t e = cudaSuccess;
	if(ctx->arena_on)
	{
		*p = arena_alloc(ctx, bytes);
		if(!*p) return AGPU_ERR_OOM;       // arena_alloc left the details in last_error
	}
	else
	{
		e = cudaMallocAsync(p, bytes, ctx->stream);
		if(e != cudaSuccess) { ctx->last_error = std::string("cudaMallocAsync: ") + cudaGetErrorString(e); cudaGetLastError(); return AGPU_ERR_OOM; }
	}
	if(zero) { e = cudaMemsetAsync(*p, 0, bytes, ctx->stream); if(e != cudaSuccess) { ctx->last_error = cudaGetErrorString(e); return AGPU_ERR_CUDA; } }
	return AGPU_OK;
}
inline void dev_free_bytes(agpu_ctx *ctx, void *p) { if(p && !ctx->arena.contains(p)) cudaFreeAsync(p, ctx->stream); }
inline void arena_destroy(agpu_ctx *ctx)
{
	for(size_t k = 0; k < ctx->arena.slabs.size(); k++) cudaFreeAsync(ctx->arena.slabs[k].base, ctx->stream);
	ctx->arena.slabs.clear(); ctx->arena.rewind();
}
// stage entry / exit of a batch: its allocations come from the arena while it owns it
struct arena_scope
{
	agpu_ctx *ctx;
	arena_scope(agpu_ctx *c, agpu_batch *b) : ctx(c) { c->arena_on = (b != NULL && c->arena_owner == b); }
	~arena_scope() { ctx->arena_on = false; }
};
#define AGPU_BATCH_SCOPE(ctx, b) arena_scope arena_scope_(ctx, b)
inline int dev_fill(agpu_ctx *ctx, void *p, int byte, size_t bytes) { if(bytes == 0) return AGPU_OK; return cudaMemsetAsync(p, byte, bytes, ctx->stream) == cudaSuccess ? AGPU_OK : AGPU_ERR_CUDA; }
inline int h2d(agpu_ctx *ctx, void *d, const void *h, size_t bytes) { if(bytes == 0) return AGPU_OK; return cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, ctx->stream) == cudaSuccess ? AGPU_OK : AGPU_ERR_CUDA; }
inline int d2h(agpu_ctx *ctx, void *h, const void *d, size_t bytes) { if(bytes == 0) return AGPU_OK; return cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, ctx->stream) == cudaSuccess ? AGPU_OK : AGPU_ERR_CUDA; }
inline int d2d(agpu_ctx *ctx, void *d, const void *s, size_t bytes) { if(bytes == 0) return AGPU_OK; return cudaMemcpyAsync(d, s, bytes, cudaMemcpyDeviceToDevice, ctx->stream) == cudaSuccess ? AGPU_OK : AGPU_ERR_CUDA; }
inline int stream_sync(agpu_ctx *ctx)
{
	cudaError_t e;
	ctx->syncs++;
	if(ctx->blocking_sync && ctx->ev_sync)
	{
		e = cudaEventRecord((cudaEvent_t)ctx->ev_sync, ctx->stream);
		if(e == cudaSuccess) e = cudaEventSynchronize((cudaEvent_t)ctx->ev_sync);
	}
	else e = cudaStreamSynchronize(ctx->stream);
	if(e != cudaSuccess) { ctx->last_error = std::string("cudaStreamSynchronize: ") + cudaGetErrorString(e); return AGPU_ERR_CUDA; }
	e = cudaGetLastError();
	if(e != cudaSuccess) { ctx->last_error = std::string("kernel launch: ") + cudaGetErrorString(e); return AGPU_ERR_CUDA; }
	return AGPU_OK;
}
inline void *pinned_alloc(size_t bytes) { void *p = NULL; if(bytes == 0) bytes = 16; if(cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return NULL; } return p; }
inline void pinned_free(void *p) { if(p) cudaFreeHost(p); }
#else
// ------------------------------------------------------------- kernel-logic test build (host)
#define CUDA_TRY(ctx, call) do { (void)(call); } while(0)
template<typename F, typename... A> inline void emu_launch(bool coop, F f, int64_t grid, unsigned block, A... a)
{
	gridDim.x = (unsigned)grid; gridDim.y = gridDim.z = 1;
	blockDim.x = coop ? 1 : block; blockDim.y = blockDim.z = 1;
	for(int64_t b = 0; b < grid; b++)
	{
		blockIdx.x = (unsigned)b; blockIdx.y = blockIdx.z = 0;
		for(unsigned t = 0; t < blockDim.x; t++)
		{
			threadIdx.x = t; threadIdx.y = threadIdx.z = 0;
			f(a...);
		}
	}
}
inline void side_fork(agpu_ctx *) {}
inline void side_join(agpu_ctx *) {}
inline void arena_destroy(agpu_ctx *) {}
struct arena_scope { arena_scope(agpu_ctx *, agpu_batch *) {} };
#define AGPU_ENTER(ctx) do {} while(0)
#define AGPU_BATCH_SCOPE(ctx, b) do {} while(0)
#define LAUNCH_T(ctx, kern, n, ...) do { int64_t n_ = (int64_t)(n); if(n_ > 0) { emu_launch(false, kern, (n_ + 255) / 256, 256, __VA_ARGS__); (ctx)->launches++; } } while(0)
#define LAUNCH_B_SIDE(ctx, kern, nblocks, nthreads, ...) LAUNCH_B(ctx, kern, nblocks, nthreads, __VA_ARGS__)
#define LAUNCH_B(ctx, kern, nblocks, nthreads, ...) do { int64_t n_ = (int64_t)(nblocks); if(n_ > 0) { emu_launch(true, kern, n_, (nthreads), __VA_ARGS__); (ctx)->launches++; } } while(0)
inline int dev_alloc_bytes(agpu_ctx *, void **p, size_t bytes, bool zero) { if(bytes == 0) bytes = 16; *p = zero ? calloc(1, bytes) : malloc(bytes); return *p ? AGPU_OK : AGPU_ERR_OOM; }
inline void dev_free_bytes(agpu_ctx *, void *p) { free(p); }
inline int dev_fill(agpu_ctx *, void *p, int byte, size_t bytes) { memset(p, byte, bytes); return AGPU_OK; }
inline int h2d(agpu_ctx *, void *d, const void *h, size_t bytes) { memcpy(d, h, bytes); return AGPU_OK; }
inline int d2h(agpu_ctx *, void *h, const void *d, size_t bytes) { memcpy(h, d, bytes); return AGPU_OK; }
inline int d2d(agpu_ctx *, void *d, const void *s, size_t bytes) { memcpy(d, s, bytes); return AGPU_OK; }
inline int stream_sync(agpu_ctx *ctx) { ctx->syncs++; return AGPU_OK; }
inline void prof_collect(agpu_ctx *) {}
inline void *pinned_alloc(size_t bytes) { return malloc(bytes ? bytes : 16); }
inline void pinned_free(void *p) { free(p); }
#endif

// ---- launch of a decoupled look-back kernel (lookback.h): kern(lb_ctl, args...) over n_tiles tiles
#define LB_STATUS_CHAINS 4
inline int lb_prepare(agpu_ctx *ctx, int64_t n_tiles, unsigned grid, unsigned long long *ticket_base, unsigned *epoch)
{
	if(n_tiles > ctx->lb_stride || ctx->lb_status == NULL || ((ctx->lb_epoch + 1) & 0x3fffu) == 0)
	{
		// (re)allocate and clear: first use, more tiles than ever before, or the 14-bit epoch is about to wrap
		int64_t stride = ctx->lb_stride > 0 ? ctx->lb_stride : ((int64_t)1 << 16);
		while(stride < n_tiles) stride *= 2;
		const size_t bytes = sizeof(unsigned long long) * (size_t)stride * LB_STATUS_CHAINS;
#ifndef AGPU_EMU
		if(stride != ctx->lb_stride || ctx->lb_status == NULL)
		{
			if(ctx->lb_status) cudaFreeAsync(ctx->lb_status, ctx->stream);
			void *p = NULL;
			if(cudaMallocAsync(&p, bytes, ctx->stream) != cudaSuccess) { cudaGetLastError(); ctx->lb_status = NULL; ctx->lb_stride = 0; return AGPU_ERR_OOM; }
			ctx->lb_status = (unsigned long long*)p;
		}
		if(cudaMemsetAsync(ctx->lb_status, 0, bytes, ctx->stream) != cudaSuccess) return AGPU_ERR_CUDA;
		if(ctx->lb_ticket == NULL)
		{
			void *p = NULL;
			if(cudaMallocAsync(&p, 64, ctx->stream) != cudaSuccess) { cudaGetLastError(); return AGPU_ERR_OOM; }
			ctx->lb_ticket = (unsigned long long*)p;
			cudaMemsetAsync(ctx->lb_ticket, 0, 64, ctx->stream);
			ctx->lb_tickets = 0;
		}
#else
		if(stride != ctx->lb_stride || ctx->lb_status == NULL) { free(ctx->lb_status); ctx->lb_status = (unsigned long long*)malloc(bytes); }
		memset(ctx->lb_status, 0, bytes);
		if(ctx->lb_ticket == NULL) { ctx->lb_ticket = (unsigned long long*)calloc(8, 8); ctx->lb_tickets = 0; }
#endif
		ctx->lb_stride = stride;
		ctx->lb_epoch = (ctx->lb_epoch + 1) & 0x3fffu;
		if(ctx->lb_epoch == 0) ctx->lb_epoch = 1;
	}
	else ctx->lb_epoch++;
	*epoch = ctx->lb_epoch & 0x3fffu;
	*ticket_base = ctx->lb_tickets;
	ctx->lb_tickets += (unsigned long long)n_tiles + grid;
	return AGPU_OK;
}
inline void lb_destroy(agpu_ctx *ctx)
{
#ifndef AGPU_EMU
	if(ctx->lb_status) cudaFreeAsync(ctx->lb_status, ctx->stream);
	if(ctx->lb_ticket) cudaFreeAsync(ctx->lb_ticket, ctx->stream);
#else
	free(ctx->lb_status); free(ctx->lb_ticket);
#endif
	ctx->lb_status = NULL; ctx->lb_ticket = NULL; ctx->lb_stride = 0;
}
#ifndef AGPU_EMU
#define LB_GRID(ctx, n_tiles) ((unsigned)((n_tiles) < (int64_t)(ctx)->sm_count * 8 ? (n_tiles) : (int64_t)(ctx)->sm_count * 8))
#define LAUNCH_LB(ctx, kern, n_tiles, ...) do { int64_t nt_ = (int64_t)(n_tiles); if(nt_ > 0) { unsigned g_ = LB_GRID(ctx, nt_); agpu::lb_ctl lc_; \
	unsigned ep_; unsigned long long tb_; TRY(lb_prepare(ctx, nt_, g_, &tb_, &ep_)); \
	lc_.status = (agpu::u64*)(ctx)->lb_status; lc_.ticket = (ctx)->lb_ticket; lc_.stride = (ctx)->lb_stride; lc_.ticket_base = tb_; lc_.epoch = ep_; \
	prof_begin(ctx, #kern); kern<<<g_, 256, 0, (ctx)->stream>>>(lc_, __VA_ARGS__); prof_end(ctx); (ctx)->launches++; } } while(0)
#else
#define LAUNCH_LB(ctx, kern, n_tiles, ...) do { int64_t nt_ = (int64_t)(n_tiles); if(nt_ > 0) { unsigned g_ = 2; agpu::lb_ctl lc_; \
	unsigned ep_; unsigned long long tb_; TRY(lb_prepare(ctx, nt_, g_, &tb_, &ep_)); \
	lc_.status = (agpu::u64*)(ctx)->lb_status; lc_.ticket = (ctx)->lb_ticket; lc_.stride = (ctx)->lb_stride; lc_.ticket_base = tb_; lc_.epoch = ep_; \
	emu_launch(true, kern, g_, 256, lc_, __VA_ARGS__); (ctx)->launches++; } } while(0)
#endif

// stream-ordered device array: owns its allocation and frees it (on the stream of the context it came from) when it goes.
// Never give one static storage duration: its destructor would run after the CUDA context is gone.
template<typename T> struct dbuf
{
	T *p = NULL;
	size_t n = 0;
	agpu_ctx *ctx = NULL;
	dbuf() = default;
	dbuf(const dbuf &) = delete;
	dbuf &operator=(const dbuf &) = delete;
	dbuf(dbuf &&o) : p(o.p), n(o.n), ctx(o.ctx) { o.p = NULL; o.n = 0; }
	dbuf &operator=(dbuf &&o)
	{
		if(this != &o) { release(); p = o.p; n = o.n; ctx = o.ctx; o.p = NULL; o.n = 0; }
		return *this;
	}
	~dbuf() { release(); }
	int alloc(agpu_ctx *c, size_t count, bool zero = false)
	{
		release();
		ctx = c;
		n = count;
		return dev_alloc_bytes(c, (void**)&p, count * sizeof(T), zero);
	}
	void release() { if(p) dev_free_bytes(ctx, p); p = NULL; n = 0; }
	int fill(agpu_ctx *c, int byte) { return dev_fill(c, p, byte, n * sizeof(T)); }
};

} // namespace agpu
inline char *agpu_pinbuf::ensure(size_t bytes)
{
	if(bytes + 1 > cap) { agpu::pinned_free(p); cap = (bytes + 1) * 5 / 4 + 64; p = (char*)agpu::pinned_alloc(cap); if(!p) cap = 0; }
	return p;
}
inline bool agpu_pinbuf::reserve_exact(size_t bytes)
{
	if(bytes <= cap) return true;
	agpu::pinned_free(p);
	cap = bytes;
	p = (char*)agpu::pinned_alloc(cap);
	if(!p) { cap = 0; return false; }
	return true;
}
inline void agpu_pinbuf::release() { agpu::pinned_free(p); p = NULL; cap = 0; }
namespace agpu {

#define TRY(x) do { int rc_ = (x); if(rc_ != AGPU_OK) return rc_; } while(0)

} // namespace agpu

#endif
