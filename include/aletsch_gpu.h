/* aletsch_gpu.h -- C ABI of the B200-native per-bundle read-evidence path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  Each entry
 * point names the reference seam it replaces (file:line under the reference tree).  The
 * library is libaletsch_gpu.so (aletsch_b200/csrc, hand-written sm_100a CUDA); there is no
 * CPU fallback: every compute entry point returns AGPU_ERR_CUDA when no device is usable.
 *
 * Unit of work: a BATCH of bundles.  The reference enters its seams once per bundle from a
 * thread pool (meta/incubator.cc:615-635); here the host packs many bundles into one
 * structure-of-arrays batch and each call processes all of them.  Device state of a batch
 * (hits, chain sets hcst/fcst, coverage map mmap, fragments, graph, clusters, bridge
 * choices) lives in HBM between calls, exactly like a `bundle` object lives between the
 * reference's calls; `agpu_*_fetch` copies a stage's results into pinned host memory and
 * hands out flat views.
 *
 * Stage map (SURVEY.md section 8):
 *   agpu_batch_evidence   bundle_base::add_hit_intervals  rnacore/bundle_base.cc:33-47,73-173
 *                         + generator::generate           meta/generator.cc:203-227
 *   agpu_batch_fragments  bundle_base::build_fragments    rnacore/bundle_base.cc:267-323
 *   agpu_batch_graph      graph_builder::build            rnacore/graph_builder.cc:24-35
 *                         + splice_graph::build_vertex_index  rnacore/splice_graph.cc:1087-1099
 *   agpu_batch_cluster    graph_cluster ctor + build_pereads_clusters  rnacore/graph_cluster.cc:13-26
 *   agpu_batch_bridge     bridge_solver ctor              bridge/bridge_solver.cc:32-46
 *   agpu_batch_update     bundle_base::update_bridges     rnacore/bundle_base.cc:420-507
 *                         as looped in bundle::bridge     meta/bundle.cc:73-79
 *   agpu_batch_bridge_all bundle::bridge                  meta/bundle.cc:55-88
 *   agpu_similarity       bundle_group::build_splice_similarity  meta/bundle_group.cc:190-231
 */
#ifndef ALETSCH_GPU_H
#define ALETSCH_GPU_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGPU_OK                 0
#define AGPU_ERR_ARG           -1   /* bad argument / call order */
#define AGPU_ERR_CUDA          -2   /* CUDA error (no device, launch failure); see agpu_last_error */
#define AGPU_ERR_OOM           -3   /* device or pinned allocation failed */
#define AGPU_ERR_INPUT         -4   /* input violates the packing contract (see agpu_batch_in) */
#define AGPU_ERR_CAPACITY      -5   /* an internal scratch bound was exceeded; nothing partial is returned */

/* library types (util/constants.h:59-62) */
#define AGPU_UNSTRANDED 0
#define AGPU_FR_FIRST   1
#define AGPU_FR_SECOND  2

typedef struct agpu_ctx agpu_ctx;       /* one per host thread / stream */
typedef struct agpu_batch agpu_batch;   /* device-resident state of one batch of bundles */

/* The values of `parameters` (util/parameters.h:19-118, defaults util/parameters.cc:19-113)
 * and `sample_profile` (rnacore/sample_profile.cc:17-33) that the path reads. */
typedef struct agpu_params
{
	int32_t library_type;                  /* sample_profile::library_type */
	int32_t min_junction_support;          /* 1 (ONT / PacBio-sub: 2) */
	int32_t normal_junction_threshold;     /* 10 */
	int32_t extend_junction_threshold;     /* 20 */
	int32_t min_subregion_gap;             /* 15 */
	int32_t min_subregion_length;          /* 15 */
	int32_t max_reads_partition_gap;       /* 10 */
	int32_t bridge_end_relaxing;           /* 10 */
	int32_t bridge_dp_solution_size;       /* 10, at most AGPU_MAX_DP_SOLUTIONS */
	int32_t bridge_dp_stack_size;          /* 5, at most AGPU_MAX_DP_STACK */
	int32_t insertsize_low;                /* sample_profile::insertsize_low, 80 until profiled */
	int32_t insertsize_high;               /* sample_profile::insertsize_high, 500 until profiled */
	int32_t max_group_size;                /* -c, 200 */
	int32_t max_num_junctions_to_combine;  /* 500 */
	double min_subregion_overlap;          /* 1.5 */
	double min_guaranteed_edge_weight;     /* 0.01 */
	double min_grouping_similarity;        /* -s, 0.10 */
	double max_grouping_similarity;        /* 0.80 */
	double min_boundary_log_ratio;         /* 2.0 (identify_boundaries, util/parameters.cc:82) */
	int32_t max_group_boundary_distance;   /* 10000 (group_start_boundaries / group_end_boundaries, util/parameters.cc:77) */
} agpu_params;

#define AGPU_MAX_DP_SOLUTIONS 16
#define AGPU_MAX_DP_STACK      8

void agpu_default_params(agpu_params *p);

/* Packed input: NB bundles, hits concatenated bundle by bundle in BAM order.
 * Packing contract (what meta/generator.cc:77-179 + bundle_base::add_hit guarantee):
 *   - within a bundle pos[] is non-decreasing (mate pairing relies on it: a hit's mate candidates are found by bisecting the
 *     bundle's pos[] for mpos; agpu_batch_fragments only runs after agpu_batch_evidence has verified the order);
 *   - no hit equals its predecessor in (pos, rpos)        (rnacore/bundle_base.cc:75-82);
 *   - rpos[i] == pos[i] + bam_cigar2rlen(cigar of i)      (rnacore/hit.cc:64);
 *   - strand[] / xs[] hold '+', '-' or '.'; all hits of a bundle share strand[]
 *     (rnacore/bundle_base.cc:100-101).
 * agpu_batch_evidence verifies these on the device and returns AGPU_ERR_INPUT if violated.
 * All arrays are caller-owned host memory (pinned memory makes the upload asynchronous).
 * BATCHING RULE.  One batch holds n_cigar < 2^32 CIGAR operations (cigar_off is 32 bits) and fewer than 2^32 - 64 coverage-window
 * positions: the sum over its bundles of (largest rpos - smallest pos + 1) rounded up to 128 (the border bitmap is indexed with
 * 32 bits).  agpu_batch_evidence returns AGPU_ERR_CAPACITY for a larger one and nothing partial is kept: cut the bundles of a
 * region batch into contiguous runs of whole bundles below both bounds -- bundles are independent (meta/bundle.cc:55-88), so the
 * cut changes no result.  bench.py: device_batches() is that cut (window estimated from the hits with 512 positions of slack per
 * bundle); the whole human genome at the depth of BASELINE configs[2] needs 4 such batches per 3 chromosomes.
 * QNAME KEYS.  qid[] stands for the query name: two hits of a bundle pair only if their keys are equal, so equal keys must mean
 * equal names INSIDE A BUNDLE.  host/bamio.cc (bam_read_records) hashes the name to 64 bits and verifies every key against a
 * 128-bit identity of the name inside the pairing window, re-keying a colliding name; a host that packs its own keys owes the
 * same guarantee (0xffffffffffffffff is reserved: AGPU_ERR_INPUT). */
typedef struct agpu_batch_in
{
	int32_t n_bundles;
	int64_t n_hits;
	int64_t n_cigar;
	const int64_t *bundle_hit_off;   /* [NB+1] */
	const int32_t *bundle_tid;       /* [NB] chromosome id */
	const int32_t *bundle_sample;    /* [NB] sample id (informational; carried through) */
	const int32_t *pos;              /* [H] hit.pos */
	const int32_t *rpos;             /* [H] hit.rpos; may be NULL: derived on the device as pos + bam_cigar2rlen (rnacore/hit.cc:64) */
	const int32_t *mpos;             /* [H] hit.mpos */
	const int32_t *isize;            /* [H] hit.isize */
	const uint16_t *flag;            /* [H] hit.flag; informational, may be NULL: no kernel reads it (the host derives strand / xs from it,
	                                    rnacore/hit.cc:106-185) and it is not uploaded */
	const uint8_t *strand;           /* [H] hit.strand; may be NULL if bundle_strand is given */
	const uint8_t *xs;               /* [H] hit.xs */
	const uint64_t *qid;             /* [H] query-name key: equal <=> same qname (rnacore/bundle_base.cc:308) */
	const uint32_t *cigar_off;       /* [H+1] into cigar[] */
	const uint32_t *cigar;           /* [n_cigar] raw BAM CIGAR ops (len<<4 | op) */
	const uint8_t *bundle_strand;    /* [NB] the strand all hits of a bundle share (rnacore/bundle_base.cc:100-101); used when strand == NULL */
} agpu_batch_in;

/* ---- context ------------------------------------------------------------------------- */
/* stream: a cudaStream_t to run on (e.g. torch's current stream), or NULL to create one. */
int agpu_create(int device, void *stream, agpu_ctx **out);
void agpu_destroy(agpu_ctx *ctx);
const char *agpu_last_error(agpu_ctx *ctx);
int agpu_sync(agpu_ctx *ctx);
/* number of times this context has waited for its stream so far (every wait drains the stream: the figure to keep low) */
int64_t agpu_sync_count(agpu_ctx *ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t agpu_launch_count(agpu_ctx *ctx);

/* Scratch arena of the context: a batch's derived state is bump-allocated from a few large slabs the context keeps.
 * agpu_reserved = bytes held now; agpu_reserve grows the arena ahead of time (e.g. to the largest size any context of a
 * stream pool has needed) so that steady-state work never allocates. */
int64_t agpu_reserved(agpu_ctx *ctx);
int agpu_reserve(agpu_ctx *ctx, int64_t bytes);

/* on = 1: agpu_batch_upload / agpu_batch_upload_packed of this context return as soon as the copies (and the decode kernels) are
 * queued on the context's stream.  The caller's host buffers must then stay untouched until the first stage call on the batch
 * has returned (every stage ends with a wait on the stream), and input errors the upload would have reported surface there.
 * This lets one host thread queue the next batch's upload on a second context before it runs the stages of the current one
 * (aletsch_b200/pipeline.py). */
int agpu_upload_async(agpu_ctx *ctx, int on);
/* how the host waits for the stream inside the stages: 0 (default) spins, lowest latency; 1 sleeps on a blocking event, for
 * boxes where the host threads of all contexts outnumber the cores */
int agpu_blocking_sync(agpu_ctx *ctx, int on);

/* optional per-kernel timing: CUDA events around every launch of this context.  agpu_profile_read
 * synchronises and writes "kernel_name\tms\tlaunches\n" lines (cumulative since the last reset). */
int agpu_profile_enable(agpu_ctx *ctx, int on);
int agpu_profile_reset(agpu_ctx *ctx);
int agpu_profile_read(agpu_ctx *ctx, char *buf, size_t cap);

/* ---- batch life cycle ---------------------------------------------------------------- */
/* host -> device copy of the packed batch (cudaMemcpyAsync per array on the ctx stream) */
int agpu_batch_upload(agpu_ctx *ctx, const agpu_batch_in *in, agpu_batch **out);
/* Compact form of the same input for the host -> device link (about 60 % of the bytes of the lean agpu_batch_in).  It
 * is decoded on the device into exactly the arrays agpu_batch_upload would have copied; every later call behaves the same.
 *   pos    : bundle_pos0[b] for a bundle's first hit, then 16-bit deltas to the previous hit (pos is non-decreasing inside a
 *            bundle); 0xFFFF announces an entry (hit index, delta) in the esc_pos list
 *   mpos   : 16-bit offset from pos; -32768 announces an entry (hit index, mpos) in esc_mpos
 *   isize  : 16 bits; -32768 announces an entry in esc_isize
 *   xs     : two bits of hit_meta[i] (bits 6-7: 0 '.', 1 '+', 2 '-')
 *   CIGAR  : bits 0-5 of hit_meta[i] 16-bit units per hit; 62 = the hit's CIGAR is the single unit default_unit (the batch's most
 *            common one-operation CIGAR, e.g. 100M) and takes no entry in units[]; 63 announces an entry (hit index, units) in
 *            esc_units; an operation of length < 4096 is one unit, the low 16 bits of its BAM encoding
 *            (len << 4 | op); a longer one (len < 2^24) is two units: 15 | (len & 0xfff) << 4, then op | (len >> 12) << 4
 *   rpos / flag / strand are not sent (see agpu_batch_in); bundle_strand is required.
 * The escape lists are sorted by hit index.  aletsch_b200/host/packer.h: packer_compact_create builds this from an
 * agpu_batch_in.  Returns AGPU_ERR_INPUT when a sentinel has no entry or the units do not decode to n_cigar operations. */
typedef struct agpu_batch_packed
{
	int32_t n_bundles;
	int64_t n_hits;
	int64_t n_cigar;                 /* CIGAR operations the units decode to */
	int64_t n_units;
	uint32_t default_unit;           /* see hit_meta */
	const int64_t *bundle_hit_off;   /* [NB+1] */
	const int32_t *bundle_tid;       /* [NB] */
	const int32_t *bundle_sample;    /* [NB] may be NULL */
	const uint8_t *bundle_strand;    /* [NB] */
	const int32_t *bundle_pos0;      /* [NB] pos of the bundle's first hit (anything for an empty bundle) */
	const uint16_t *dpos;            /* [H] */
	const int16_t *dmpos;            /* [H] */
	const int16_t *isize16;          /* [H] */
	const uint64_t *qid;             /* [H] */
	const uint8_t *hit_meta;         /* [H] */
	const uint16_t *units;           /* [n_units] */
	int64_t n_esc_pos, n_esc_mpos, n_esc_isize, n_esc_units;
	const int64_t *esc_pos_idx, *esc_mpos_idx, *esc_isize_idx, *esc_units_idx;
	const int32_t *esc_pos_val, *esc_mpos_val, *esc_isize_val, *esc_units_val;
} agpu_batch_packed;
int agpu_batch_upload_packed(agpu_ctx *ctx, const agpu_batch_packed *in, agpu_batch **out);
/* same, but the arrays of `in` are DEVICE pointers already resident in HBM (no copy) */
int agpu_batch_adopt(agpu_ctx *ctx, const agpu_batch_in *in_device, agpu_batch **out);
void agpu_batch_free(agpu_ctx *ctx, agpu_batch *b);
/* forget all derived state (chains, coverage, fragments, graph ...) but keep the uploaded hits */
int agpu_batch_reset(agpu_ctx *ctx, agpu_batch *b);
/* A new batch holding n_sel bundles taken from existing batches: bundle k of *out is bundle sel_bundle[k] of src[sel_src[k]],
 * copied device to device (aletsch_b200/clusters.py uses it to cut a job a second time, by cross-sample cluster, without sending
 * the hits over PCIe again).  The output is a fresh batch like the result of agpu_batch_upload: it owns copies of bundle_hit_off,
 * pos, rpos, mpos, isize, xs, qid, cigar_off and cigar on the device, bundle_tid and bundle_sample on the host, and no derived
 * state.  strand is always per hit (a source uploaded with bundle_strand only has that strand expanded to its hits); rpos is the
 * source's device array, uploaded or derived; bundle_sample is kept only if every source has it; flag is not carried (no kernel
 * reads it).  A bundle may be selected more than once; n_sel == 0 gives a valid empty batch.
 * Sources may come from any upload entry or agpu_batch_adopt and may belong to other contexts on the same device as ctx: the call
 * orders itself after the work already queued on each source's context stream (device-side event waits) and ends with a stream
 * synchronisation, after which the sources may be reset or freed.  No other call may run on a source while the gather runs.
 * Errors: AGPU_ERR_ARG for an index out of range, a NULL source, a source on another device or a source with coverage edits
 * (agpu_batch_coverage_edit: per-hit state that is not regrouped); AGPU_ERR_CAPACITY when the output would hold 2^32 or more CIGAR
 * operations (cigar_off is 32 bits).  Nothing partial is kept on any error.  The packing contract is not checked here: a
 * violation in a selected bundle surfaces at the output's agpu_batch_evidence, as it would have in the source. */
int agpu_batch_gather(agpu_ctx *ctx, int32_t n_src, agpu_batch *const *src, int32_t n_sel, const int32_t *sel_src, const int32_t *sel_bundle,
		agpu_batch **out);
/* The input columns the stages read, as DEVICE pointers, with the batch's counts: bundle_hit_off, pos, rpos, mpos, isize, strand
 * (per hit) or bundle_strand (per bundle; the other one is NULL), xs, qid, cigar_off and cigar.  bundle_tid, bundle_sample and
 * flag are returned as NULL: the first two live on the host side of the batch, flag is never uploaded.  rpos is the uploaded or
 * the derived array.  A batch built by agpu_batch_gather always has rpos and a per-hit strand.  No stage writes these arrays, so
 * the pointers stay valid and unchanged until agpu_batch_free, e.g. as send buffers of a transfer between GPUs
 * (aletsch_b200/shard.py), while stages run on the batch.  Builds without a device (the kernel-logic emulation) return host
 * pointers.  AGPU_ERR_ARG for NULL arguments. */
int agpu_batch_inputs(agpu_ctx *ctx, agpu_batch *b, agpu_batch_in *out);

/* ---- stages (asynchronous on the ctx stream unless noted) ----------------------------- */
int agpu_batch_evidence(agpu_ctx *ctx, agpu_batch *b, const agpu_params *p);
int agpu_batch_fragments(agpu_ctx *ctx, agpu_batch *b);
int agpu_batch_graph(agpu_ctx *ctx, agpu_batch *b, const agpu_params *p);
int agpu_batch_cluster(agpu_ctx *ctx, agpu_batch *b, const agpu_params *p);
int agpu_batch_bridge(agpu_ctx *ctx, agpu_batch *b, const agpu_params *p);
int agpu_batch_update(agpu_ctx *ctx, agpu_batch *b);
/* evidence (if not done) + fragments (if not done) + graph + cluster + bridge + update */
int agpu_batch_bridge_all(agpu_ctx *ctx, agpu_batch *b, const agpu_params *p);

/* ---- results: flat views into ctx-owned pinned host memory, valid until the next fetch
 *      of the same kind on this batch or agpu_batch_free.  Each fetch synchronises. ------ */

typedef struct agpu_chainset_view       /* chain_set (rnacore/chain_set.h:18-35), insertion-ordered */
{
	const int32_t *bundle_chain_off;    /* [NB+1] chains of bundle b: [off[b], off[b+1]) */
	const int32_t *chain_off;           /* [C+1] into chain_val */
	const int32_t *chain_val;           /* splice coordinates l0 r0 l1 r1 ... */
	const int32_t *chain_cnt;           /* [3C] n. n+ n-  (AI3) */
	const int32_t *chain_grp;           /* [C] index i of chains[i][j] inside its bundle */
	const int32_t *handle_chain;        /* [H or F] bundle-local chain index of hit / fragment, -1 if none (hmap) */
	int64_t n_chains;
	int64_t n_handles;
} agpu_chainset_view;

typedef struct agpu_evidence_view
{
	int32_t n_bundles;
	const int32_t *lpos;                /* [NB] bundle_base::lpos */
	const int32_t *rpos;                /* [NB] bundle_base::rpos */
	const uint8_t *strand;              /* [NB] bundle_base::strand after compute_strand */
	const int64_t *seg_off;             /* [NB+1] */
	const int32_t *seg;                 /* [3S] l r cov: split_interval_map mmap in order */
	const int64_t *splice_off;          /* [NB+1] */
	const int32_t *splices;             /* bundle_base::splices (sorted unique) */
	agpu_chainset_view hcst;
} agpu_evidence_view;

typedef struct agpu_fragments_view
{
	const int64_t *frg_off;             /* [NB+1] */
	const int32_t *frgs;                /* [3F] h1 h2 type, h bundle-local; bundle_base::frgs in order */
	agpu_chainset_view fcst;            /* handles are bundle-local fragment indices */
	const int32_t *bridged;             /* [NB] sum of update_bridges return values so far */
} agpu_fragments_view;

typedef struct agpu_graph_view
{
	const int32_t *junc_off;            /* [NB+1] */
	const int32_t *junc;                /* [9J] lpos rpos count xs0 xs1 xs2 strand lexon rexon (graph_builder::junctions order) */
	const int32_t *pexon_off;           /* [NB+1] */
	const int32_t *pexon;               /* [5P] lpos rpos ltype rtype regional */
	const double *pexon_d;              /* [4P] ave dev max pvalue (max = -1 for the 1-bp stubs, which the reference leaves unset) */
	const int32_t *vert_off;            /* [NB+1]; V = P + 2 per bundle */
	const int32_t *vert;                /* [5V] lpos rpos length type regional */
	const double *vert_d;               /* [3V] weight stddev maxcov */
	const int32_t *edge_off;            /* [NB+1] */
	const int32_t *edge;                /* [3E] src dst strand, in the reference's insertion order; removed edges have src = -1 */
	const double *edge_d;               /* [E] weight */
	const uint8_t *strand;              /* [NB] splice_graph::strand */
} agpu_graph_view;

typedef struct agpu_cluster_view        /* vector<pereads_cluster> per bundle, in order */
{
	const int64_t *clu_off;             /* [NB+1] */
	const int32_t *bounds;              /* [4C] */
	const int32_t *extend;              /* [4C] */
	const int32_t *count;               /* [C] */
	const int32_t *chain1;              /* [C] bundle-local hcst chain index of chain1, -1 if empty */
	const int32_t *chain2;              /* [C] */
	const int64_t *frlist_off;          /* [C+1] */
	const int32_t *frlist;              /* bundle-local fragment indices */
	int64_t n_clusters;
} agpu_cluster_view;

typedef struct agpu_bridge_view         /* bridge_solver::opt per cluster */
{
	const int32_t *type;                /* [C] -1 / 1 / 2 */
	const int32_t *strand;              /* [C] */
	const int32_t *choices;             /* [C] */
	const double *score;                /* [C] */
	const int64_t *chain_off;           /* [C+1] */
	const int32_t *chain;
	const int64_t *whole_off;           /* [C+1] */
	const int32_t *whole;
} agpu_bridge_view;

int agpu_evidence_fetch(agpu_ctx *ctx, agpu_batch *b, agpu_evidence_view *v);
/* only bundle::splices (sorted unique splice positions per bundle): splice_off[NB+1], splices[] */
int agpu_splices_fetch(agpu_ctx *ctx, agpu_batch *b, const int64_t **splice_off, const int32_t **splices);
int agpu_fragments_fetch(agpu_ctx *ctx, agpu_batch *b, agpu_fragments_view *v);
int agpu_graph_fetch(agpu_ctx *ctx, agpu_batch *b, agpu_graph_view *v);
int agpu_cluster_fetch(agpu_ctx *ctx, agpu_batch *b, agpu_cluster_view *v);
int agpu_bridge_fetch(agpu_ctx *ctx, agpu_batch *b, agpu_bridge_view *v);

/* Everything bundle::bridge leaves behind (meta/bundle.cc:55-88), in one call: the bundle_base members it updates (mmap, hcst,
 * frgs, fcst: evidence + fragments views) and its locals (splice_graph gr, vector<pereads_cluster> vc, bridge_solver::opt:
 * graph, cluster and bridge views), packed on the device and copied into the context's pinned buffers.  `what` selects the
 * views; `bytes` returns the device -> host bytes this call copied.  The views stay valid until the next fetch of the same
 * kind on this context. */
#define AGPU_RESULT_EVIDENCE  1u
#define AGPU_RESULT_FRAGMENTS 2u
#define AGPU_RESULT_GRAPH     4u
#define AGPU_RESULT_CLUSTERS  8u
#define AGPU_RESULT_BRIDGES  16u
#define AGPU_RESULT_ALL      31u
typedef struct agpu_results
{
	agpu_evidence_view evidence;
	agpu_fragments_view fragments;
	agpu_graph_view graph;
	agpu_cluster_view clusters;
	agpu_bridge_view bridges;
	int64_t bytes;
} agpu_results;
int agpu_batch_results(agpu_ctx *ctx, agpu_batch *b, uint32_t what, agpu_results *out);
/* Pinned result buffers belong to the context and grow on demand (a pinned allocation synchronises the device).  A pool of
 * contexts that share a queue of batches calls this after a warm-up pass so that every context's buffers are at least as large
 * as the largest any of them has needed: dst's buffers grow to src's sizes, nothing shrinks.  Both contexts must be idle. */
int agpu_pinned_match(agpu_ctx *dst, agpu_ctx *src);
/* device -> host bytes the fetches of this context have copied so far */
int64_t agpu_d2h_bytes(agpu_ctx *ctx);

/* counters of the batch (host copies, synchronises): hits, cigar ops, coverage span L,
 * segments S, chains, junctions J, vertices V, edges E, fragments F, clusters C, bridged pairs */
typedef struct agpu_counts
{
	int64_t hits, cigar_ops, span, segments, chains, splice_ints, junctions, vertices, edges;
	int64_t fragments, clusters, bridged, piers;
	int64_t borders, cluster_members, bridge_chain_ints, bridge_whole_ints;   /* ranked coverage borders, sum of frlist sizes, sizes of opt[].chain / opt[].whole */
	int64_t big_group_members;   /* of cluster_members: those in fragment groups of more than 16 (partitioned by a warp each, not a thread) */
} agpu_counts;
int agpu_batch_counts(agpu_ctx *ctx, agpu_batch *b, agpu_counts *c);
/* per bundle: out[4k..4k+3] = coverage segments (0 while the coverage map awaits its rebuild after agpu_batch_update), fragments,
 * paired-read clusters, bridged pairs (sum of the update_bridges return values, rnacore/bundle_base.cc:460) */
int agpu_batch_bundle_counts(agpu_ctx *ctx, agpu_batch *b, int64_t *out);

/* ---- stage 5: junction-set similarity ------------------------------------------------ */
/* G sorted splice lists (bundle::splices); for every pair i<j: c = |splices_i ∩ splices_j| and
 * r = c / min(|splices_i|, |splices_j|).  out_c / out_r are dense G x G (row-major, upper
 * triangle filled, diagonal and lower triangle 0), caller-owned host memory. */
int agpu_similarity(agpu_ctx *ctx, int32_t n_lists, const int64_t *list_off, const int32_t *list_val,
		int32_t *out_c, double *out_r);

/* diagnostic: the permutation std::sort(v.begin(), v.end(), [](a, b){ return key[a] < key[b]; }) leaves on v = 0..n-1, as
 * computed by the device's re-implementation of libstdc++'s introsort (one thread for n <= 48, a whole warp above).  Used by
 * the tests to pin the tie order that leaks into pereads_cluster::bounds (rnacore/graph_cluster.cc:183-186). */
int agpu_debug_sort_perm(agpu_ctx *ctx, const int32_t *keys, int32_t n, int32_t *perm_out);

/* bundle_group::resolve (meta/bundle_group.cc:26-56) over G bundles given by their sorted splice lists: splice-position
 * inverted index, two rounds (max_grouping_similarity, then min_grouping_similarity) of size-capped single-linkage with the
 * pairwise similarities taken from the device (agpu_similarity).  out_group_of[i] = group of bundle i, groups numbered in
 * first-member order like bundle_group::gvv (build_groups, :320-342).  The unions follow the reference's order: pairs of one
 * splice position sorted by r descending with std::sort (ties as libstdc++ leaves them). */
int agpu_group_resolve(agpu_ctx *ctx, int32_t n_lists, const int64_t *list_off, const int32_t *list_val, const agpu_params *p,
		int32_t *out_group_of, int32_t *out_n_groups);

/* ---- phasing paths: bundle_base::build_phase_set (rnacore/bundle_base.cc:338-418) against the bundles' current splice
 * graphs (those of the last agpu_batch_graph, i.e. transform(bd, gr, false)).  Every bridged fragment and every hit outside a
 * paired fragment contributes [lpos(vertex of its start), intron chain ..., rpos(vertex of its end)] when non-decreasing;
 * equal lists are counted (phase_set::add, rnacore/phase_set.cc:12-25).  The view lists the distinct coordinate lists of every
 * bundle in the order of phase_set::pmap (lexicographic). */
typedef struct agpu_phase_view
{
	const int64_t *phase_off;           /* [NB+1] phases of bundle b: [off[b], off[b+1]) */
	const int64_t *coord_off;           /* [P+1] into coords */
	const int32_t *coords;              /* exon coordinate lists (even length) */
	const int32_t *count;               /* [P] multiplicity */
	int64_t n_phases;
} agpu_phase_view;
int agpu_batch_phase_set(agpu_ctx *ctx, agpu_batch *b);
int agpu_phase_fetch(agpu_ctx *ctx, agpu_batch *b, agpu_phase_view *v);

/* ---- boundary revision: the revising half of assembler::transform(bd, gr, true) (meta/assembler.cc:930-944) on the bundles'
 * own splice graphs.  identify_boundaries (rnacore/graph_reviser.cc:1068-1283) adds a start edge 0 -> a / an end edge b -> n
 * wherever log(2 + maxcov) / log(2 + weight entering / leaving) of a continuous run of vertices reaches
 * min_boundary_log_ratio, best ratio first, until none is left; remove_false_boundaries (:1285-1377) then records, for the
 * vertices that carry an end (start) edge, how many paired fragments that are still unbridged (type 0) leave (enter) there,
 * and log(1 + count + w) - log(1 + w).  The graph keeps its vertices, so locate_vertex and the phase set are unaffected; the
 * refine_splice_graph that follows in the reference removes nothing.  Call after agpu_batch_graph and the bridging calls.
 * The view lists, per bundle, the added edges in the order the reference adds them (src dst, vertex numbers of
 * agpu_graph_view) with their weights, and the four annotations of every vertex. */
typedef struct agpu_revise_view
{
	const int64_t *edge_off;            /* [NB+1] */
	const int32_t *edge;                /* [2E'] src dst */
	const double *edge_w;               /* [E'] maxcov - entering (leaving) weight */
	const int64_t *vert_off;            /* [NB+1]; V = P + 2 per bundle */
	const int32_t *unbridge;            /* [2V] unbridge_leaving_count unbridge_coming_count (rnacore/vertex_info.h:38-41) */
	const double *unbridge_ratio;       /* [2V] unbridge_leaving_ratio unbridge_coming_ratio */
	int64_t n_edges, n_vertices;
} agpu_revise_view;
int agpu_batch_revise(agpu_ctx *ctx, agpu_batch *b, const agpu_params *p);
int agpu_revise_fetch(agpu_ctx *ctx, agpu_batch *b, agpu_revise_view *v);

/* ---- group-level re-bridge: assembler::bridge (meta/assembler.cc:977-1018) for many clusters of bundles at once ----
 * Cluster g holds the bundles group_bundles[group_off[g] .. group_off[g+1]) in the order of the reference's `gv` (>= 2
 * members of one chromosome and strand; a bundle may appear in at most one cluster).  Per cluster: the members are merged
 * into a combined bundle in the order of combine_bundles (descending segment count, std::sort; meta/assembler.cc:152-175) --
 * chain sets added, coverage maps added, bounds joined (bundle::combine, meta/bundle.cc:90-107) --, its splice graph is built
 * (transform(cb, gr, false), meta/assembler.cc:930-944), and every member is clustered, bridged and updated against that
 * graph (graph_cluster, bridge_solver, update_bridges).  Needs evidence and fragments of the batch (normally after
 * agpu_batch_bridge_all).  Afterwards the fragments / fcst / coverage of the member bundles are updated, and
 * agpu_cluster_fetch / agpu_bridge_fetch describe this pass (bundles outside every cluster have no clusters). */
int agpu_batch_group_bridge(agpu_ctx *ctx, agpu_batch *b, int32_t n_groups, const int32_t *group_off, const int32_t *group_bundles,
		const agpu_params *p);
/* the combined bundles of the last agpu_batch_group_bridge, one per cluster: evidence view (bounds, strand, mmap, splices,
 * combined hcst; its handles are the member chains in combine order), combined fcst, splice graph, and the combine order of
 * the members (flattened like group_bundles).  Any of the outputs may be NULL. */
int agpu_group_fetch(agpu_ctx *ctx, agpu_batch *b, agpu_evidence_view *cev, agpu_chainset_view *cfcst, agpu_graph_view *cgr,
		const int32_t **combine_order);

/* ---- insert-size preview: previewer::infer_insertsize (meta/previewer.cc:151-304) ----
 * The host runs the record loop (aletsch_b200/host/packer.h: packer_preview_add) and uploads the preview bundles like any batch.
 * Two things make the reference's preview bundles differ from ordinary ones, both consequences of bundle_base::interval_buf
 * (rnacore/bundle_base.cc:106-204: the previewer never flushes it and clear() does not reset it); agpu_batch_coverage_edit hands
 * them to the device before the evidence stage:
 *   skip_mblocks[H]   bit z set: the z-th BAM_CMATCH operation of the hit adds no coverage (it is still in the buffer when
 *                     previewer::process looks at the bundle); may be NULL
 *   extra intervals   (bundle, l, r, count): blocks of an earlier bundle flushed into this one's map (matters after a
 *                     chromosome change only); clipped to the bundle's coverage window
 * agpu_batch_preview then is previewer::process for every bundle of the batch: build_fragments, graph_builder::build,
 * graph_cluster with a partition gap of 2, and per paired-read cluster the fragment length the previewer enters into its
 * histogram (INT32_MIN where it enters none).  The cap of 1000 clusters per bundle, the break at max_preview_reads and the
 * percentiles are the host's (packer_insertsize_profile). */
typedef struct agpu_preview_view
{
	const int64_t *clu_off;             /* [NB + 1] clusters of bundle b in vector<pereads_cluster> order */
	const int32_t *isize;               /* [C] bounds[3] - bounds[0] - intron length, or INT32_MIN */
	int64_t n_clusters;
} agpu_preview_view;
int agpu_batch_coverage_edit(agpu_ctx *ctx, agpu_batch *b, const uint16_t *skip_mblocks, int64_t n_extra, const int32_t *extra_bundle,
		const int32_t *extra_l, const int32_t *extra_r, const int32_t *extra_count);
int agpu_batch_preview(agpu_ctx *ctx, agpu_batch *b, const agpu_params *p);
int agpu_preview_fetch(agpu_ctx *ctx, agpu_batch *b, agpu_preview_view *v);

/* ---- cross-sample support features: the support passes of assembler::assemble(vector<bundle*>) (meta/assembler.cc:177-373) ----
 * For every cluster (same layout as agpu_batch_group_bridge; members in the order of the reference's `gv`; bundle_sample is
 * required): the members' graphs are rebuilt and revised (transform(bd, gr, true), meta/assembler.cc:930-944), the updated
 * members are combined again and the combined graph gx built (transform(bx, gx, false), :190-203), every edge starts with its
 * own sample and weight and the junctions are entered into the cluster's junction -> samples map (:205-293); then, member by
 * member in order: junction_support (:375-417), and against every member j of the cluster start_end_support (:678-779),
 * non_splicing_support (:419-462) and boundary_extend for the three position types (:781-880), then the same against gx; gx
 * itself collects start_end / non_splicing support from every member and finally its junction support (:296-330).
 * ORDER: the reference assembles member k right after its own round, and assemble(gr, ps, sid) (:1075-1134) regroups the start /
 * end boundaries of k's graph (group_start_boundaries / group_end_boundaries, rnacore/graph_reviser.cc:916-1066) -- so the
 * members after k see k's graph regrouped; that is reproduced.  It then hands the graph to scallop BY REFERENCE, which
 * decomposes it in place; what the later members would read out of a decomposed graph is NOT reproduced here (it cannot be
 * without running scallop between the rounds): a host that needs it calls this once per cluster prefix, or -- equivalently for
 * member 0 and for every cluster whose members do not overlap -- uses these rows as they are.  The parity tests compare
 * against the reference's own functions driven in this order (oracle/ref_driver.cc: ref_group_support, ORC_SUPPORT_GROUP_ONLY).
 * Call after agpu_batch_bridge_all and agpu_batch_group_bridge.  The member graphs of the batch (agpu_graph_fetch,
 * agpu_revise_fetch) and the combined graphs (agpu_group_fetch) afterwards describe the graphs the rows refer to.
 * Returns AGPU_ERR_CAPACITY when the (edge x sample) scratch of the clusters passed in one call exceeds 12 GB: split the list. */
typedef struct agpu_support_view
{
	int32_t n_graphs;                   /* the members of all clusters in the caller's order, then one combined graph per cluster */
	const int64_t *vert_off;            /* [n_graphs + 1] */
	const double *loss;                 /* [4V] vertex_info::boundary_loss1, 2, 3, boundary_merged_loss */
	const int64_t *edge_off;            /* [n_graphs + 1]; edges of a graph in (source, target) order, added boundary edges included */
	const int32_t *edge;                /* [3E] source target edge_info::count */
	const double *abd;                  /* [E] edge_info::abd */
	const int64_t *sample_off;          /* [E + 1] */
	const int32_t *sample;              /* edge_info::samples = keys of edge_info::spAbd, ascending; -1 is the combined graph */
	const double *sample_abd;           /* edge_info::spAbd values */
} agpu_support_view;
int agpu_batch_group_support(agpu_ctx *ctx, agpu_batch *b, int32_t n_groups, const int32_t *group_off, const int32_t *group_bundles,
		const agpu_params *p);
int agpu_support_fetch(agpu_ctx *ctx, agpu_batch *b, agpu_support_view *v);

/* The same for MANY bundle groups in one call (one group per (chromosome, region, strand), meta/incubator.cc:461-471):
 * group g owns the lists [group_off[g], group_off[g + 1]).  agpu_similarity_batch fills, for every group, a dense G x G
 * matrix of pair counts at out_c + c_off[g] (c_off[n_groups] = total); groups of up to 192 lists are resolved by one CTA
 * each in a single launch, larger ones by the tiled kernels.  agpu_group_resolve_batch adds the host control flow of
 * bundle_group::resolve per group: out_group_of[l] is the cluster of list l inside its bundle group. */
int agpu_similarity_batch(agpu_ctx *ctx, int32_t n_groups, const int32_t *group_off, const int64_t *list_off, const int32_t *list_val,
		const int64_t *c_off, int32_t *out_c);
int agpu_group_resolve_batch(agpu_ctx *ctx, int32_t n_groups, const int32_t *group_off, const int64_t *list_off, const int32_t *list_val,
		const agpu_params *p, int32_t *out_group_of, int32_t *out_n_groups);

#ifdef __cplusplus
}
#endif
#endif
