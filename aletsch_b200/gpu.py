"""ctypes binding of the C ABI in include/aletsch_gpu.h (libaletsch_gpu.so, hand-written sm_100a CUDA).

No fallback: importing is cheap, but ``Context()`` raises if the CUDA library is missing or no
device is usable.  The kernel-logic test tier may pass ``lib_path`` of the host emulation build
(tests/emu) explicitly; nothing in the product selects it.
"""
import ctypes as C
import os
import numpy as np

from .hostlib import BatchIn

_HERE = os.path.dirname(os.path.abspath(__file__))
GPU_SO = os.path.join(_HERE, "libaletsch_gpu.so")


class Params(C.Structure):
    """agpu_params"""
    _fields_ = [("library_type", C.c_int32), ("min_junction_support", C.c_int32), ("normal_junction_threshold", C.c_int32),
                ("extend_junction_threshold", C.c_int32), ("min_subregion_gap", C.c_int32), ("min_subregion_length", C.c_int32),
                ("max_reads_partition_gap", C.c_int32), ("bridge_end_relaxing", C.c_int32),
                ("bridge_dp_solution_size", C.c_int32), ("bridge_dp_stack_size", C.c_int32), ("insertsize_low", C.c_int32),
                ("insertsize_high", C.c_int32), ("max_group_size", C.c_int32), ("max_num_junctions_to_combine", C.c_int32),
                ("min_subregion_overlap", C.c_double), ("min_guaranteed_edge_weight", C.c_double),
                ("min_grouping_similarity", C.c_double), ("max_grouping_similarity", C.c_double),
                ("min_boundary_log_ratio", C.c_double), ("max_group_boundary_distance", C.c_int32)]


P32 = C.POINTER(C.c_int32)
P64 = C.POINTER(C.c_int64)
PF = C.POINTER(C.c_double)
PU8 = C.POINTER(C.c_uint8)


class ChainsetView(C.Structure):
    _fields_ = [("bundle_chain_off", P32), ("chain_off", P32), ("chain_val", P32), ("chain_cnt", P32), ("chain_grp", P32),
                ("handle_chain", P32), ("n_chains", C.c_int64), ("n_handles", C.c_int64)]


class EvidenceView(C.Structure):
    _fields_ = [("n_bundles", C.c_int32), ("lpos", P32), ("rpos", P32), ("strand", PU8), ("seg_off", P64), ("seg", P32),
                ("splice_off", P64), ("splices", P32), ("hcst", ChainsetView)]


class FragmentsView(C.Structure):
    _fields_ = [("frg_off", P64), ("frgs", P32), ("fcst", ChainsetView), ("bridged", P32)]


class GraphView(C.Structure):
    _fields_ = [("junc_off", P32), ("junc", P32), ("pexon_off", P32), ("pexon", P32), ("pexon_d", PF), ("vert_off", P32),
                ("vert", P32), ("vert_d", PF), ("edge_off", P32), ("edge", P32), ("edge_d", PF), ("strand", PU8)]


class ClusterView(C.Structure):
    _fields_ = [("clu_off", P64), ("bounds", P32), ("extend", P32), ("count", P32), ("chain1", P32), ("chain2", P32),
                ("frlist_off", P64), ("frlist", P32), ("n_clusters", C.c_int64)]


class BridgeView(C.Structure):
    _fields_ = [("type", P32), ("strand", P32), ("choices", P32), ("score", PF), ("chain_off", P64), ("chain", P32),
                ("whole_off", P64), ("whole", P32)]


class Results(C.Structure):
    """agpu_results"""
    _fields_ = [("evidence", EvidenceView), ("fragments", FragmentsView), ("graph", GraphView), ("clusters", ClusterView),
                ("bridges", BridgeView), ("bytes", C.c_int64)]


RESULT_EVIDENCE, RESULT_FRAGMENTS, RESULT_GRAPH, RESULT_CLUSTERS, RESULT_BRIDGES, RESULT_ALL = 1, 2, 4, 8, 16, 31


class SupportView(C.Structure):
    _fields_ = [("n_graphs", C.c_int32), ("vert_off", P64), ("loss", PF), ("edge_off", P64), ("edge", P32), ("abd", PF),
                ("sample_off", P64), ("sample", P32), ("sample_abd", PF)]


class PreviewView(C.Structure):
    _fields_ = [("clu_off", P64), ("isize", P32), ("n_clusters", C.c_int64)]


class ReviseView(C.Structure):
    _fields_ = [("edge_off", P64), ("edge", P32), ("edge_w", PF), ("vert_off", P64), ("unbridge", P32), ("unbridge_ratio", PF),
                ("n_edges", C.c_int64), ("n_vertices", C.c_int64)]


class PhaseView(C.Structure):
    _fields_ = [("phase_off", P64), ("coord_off", P64), ("coords", P32), ("count", P32), ("n_phases", C.c_int64)]


class Counts(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("hits", "cigar_ops", "span", "segments", "chains", "splice_ints", "junctions", "vertices",
                                         "edges", "fragments", "clusters", "bridged", "piers", "borders", "cluster_members",
                                         "bridge_chain_ints", "bridge_whole_ints", "big_group_members")]


ABI_SYMBOLS = ["agpu_default_params", "agpu_create", "agpu_destroy", "agpu_last_error", "agpu_sync", "agpu_launch_count", "agpu_sync_count",
               "agpu_batch_upload", "agpu_batch_adopt", "agpu_batch_free", "agpu_batch_reset", "agpu_batch_evidence",
               "agpu_batch_fragments", "agpu_batch_graph", "agpu_batch_cluster", "agpu_batch_bridge", "agpu_batch_update",
               "agpu_batch_bridge_all", "agpu_evidence_fetch", "agpu_fragments_fetch", "agpu_graph_fetch", "agpu_cluster_fetch",
               "agpu_bridge_fetch", "agpu_batch_counts", "agpu_similarity", "agpu_profile_enable", "agpu_profile_reset",
               "agpu_profile_read", "agpu_group_resolve", "agpu_debug_sort_perm", "agpu_similarity_batch", "agpu_group_resolve_batch", "agpu_splices_fetch", "agpu_batch_bundle_counts",
               "agpu_batch_group_bridge", "agpu_group_fetch", "agpu_batch_phase_set", "agpu_phase_fetch", "agpu_batch_revise", "agpu_revise_fetch", "agpu_batch_upload_packed", "agpu_reserved", "agpu_reserve", "agpu_blocking_sync", "agpu_upload_async",
               "agpu_batch_results", "agpu_d2h_bytes", "agpu_pinned_match",
               "agpu_batch_group_support", "agpu_support_fetch", "agpu_batch_coverage_edit", "agpu_batch_preview", "agpu_preview_fetch",
               "agpu_batch_gather", "agpu_batch_inputs"]


def load(lib_path=None):
    # ALETSCH_GPU_LIB: another build of the same sources (e.g. a tuning variant under test); never a different implementation
    path = lib_path or os.environ.get("ALETSCH_GPU_LIB") or GPU_SO
    if not os.path.exists(path):
        raise RuntimeError("CUDA library %s is missing: run __graft_entry__.build() (there is no CPU fallback)" % path)
    L = C.CDLL(path)
    L.agpu_create.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
    L.agpu_destroy.argtypes = [C.c_void_p]
    L.agpu_last_error.restype = C.c_char_p
    L.agpu_last_error.argtypes = [C.c_void_p]
    L.agpu_sync.argtypes = [C.c_void_p]
    L.agpu_launch_count.restype = C.c_int64
    L.agpu_launch_count.argtypes = [C.c_void_p]
    L.agpu_sync_count.restype = C.c_int64
    L.agpu_sync_count.argtypes = [C.c_void_p]
    L.agpu_default_params.argtypes = [C.POINTER(Params)]
    L.agpu_reserved.restype = C.c_int64
    L.agpu_reserved.argtypes = [C.c_void_p]
    L.agpu_reserve.argtypes = [C.c_void_p, C.c_int64]
    L.agpu_blocking_sync.argtypes = [C.c_void_p, C.c_int]
    L.agpu_upload_async.argtypes = [C.c_void_p, C.c_int]
    L.agpu_batch_upload.argtypes = [C.c_void_p, C.POINTER(BatchIn), C.POINTER(C.c_void_p)]
    L.agpu_batch_adopt.argtypes = [C.c_void_p, C.POINTER(BatchIn), C.POINTER(C.c_void_p)]
    L.agpu_batch_upload_packed.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
    L.agpu_batch_gather.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
    L.agpu_batch_inputs.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(BatchIn)]
    L.agpu_batch_free.argtypes = [C.c_void_p, C.c_void_p]
    L.agpu_batch_reset.argtypes = [C.c_void_p, C.c_void_p]
    for n in ("evidence", "graph", "cluster", "bridge", "bridge_all"):
        getattr(L, "agpu_batch_" + n).argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Params)]
    for n in ("fragments", "update"):
        getattr(L, "agpu_batch_" + n).argtypes = [C.c_void_p, C.c_void_p]
    L.agpu_evidence_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(EvidenceView)]
    L.agpu_fragments_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(FragmentsView)]
    L.agpu_graph_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(GraphView)]
    L.agpu_cluster_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(ClusterView)]
    L.agpu_bridge_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(BridgeView)]
    L.agpu_batch_counts.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Counts)]
    L.agpu_batch_results.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(Results)]
    L.agpu_d2h_bytes.restype = C.c_int64
    L.agpu_d2h_bytes.argtypes = [C.c_void_p]
    L.agpu_pinned_match.argtypes = [C.c_void_p, C.c_void_p]
    L.agpu_splices_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(P64), C.POINTER(P32)]
    L.agpu_batch_bundle_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.agpu_batch_phase_set.argtypes = [C.c_void_p, C.c_void_p]
    L.agpu_phase_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(PhaseView)]
    L.agpu_batch_revise.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Params)]
    L.agpu_revise_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(ReviseView)]
    L.agpu_batch_group_bridge.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(Params)]
    L.agpu_batch_group_support.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(Params)]
    L.agpu_support_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(SupportView)]
    L.agpu_batch_coverage_edit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.agpu_batch_preview.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Params)]
    L.agpu_preview_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(PreviewView)]
    L.agpu_group_fetch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(EvidenceView), C.POINTER(ChainsetView), C.POINTER(GraphView), C.POINTER(P32)]
    L.agpu_similarity.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.agpu_group_resolve.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(Params), C.c_void_p, C.c_void_p]
    L.agpu_debug_sort_perm.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    L.agpu_similarity_batch.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.agpu_group_resolve_batch.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Params), C.c_void_p, C.c_void_p]
    L.agpu_profile_enable.argtypes = [C.c_void_p, C.c_int]
    L.agpu_profile_reset.argtypes = [C.c_void_p]
    L.agpu_profile_read.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t]
    L.host_memory = hasattr(L, "agpu_emu_build")      # the kernel-logic emulation build (tests/emu): its "device" arrays are host memory
    return L


def default_params(**kw):
    p = Params()
    # defaults of util/parameters.cc:19-113; filled by the library itself when loadable, else statically
    p.library_type, p.min_junction_support, p.normal_junction_threshold, p.extend_junction_threshold = 1, 1, 10, 20
    p.min_subregion_gap, p.min_subregion_length, p.max_reads_partition_gap, p.bridge_end_relaxing = 15, 15, 10, 10
    p.bridge_dp_solution_size, p.bridge_dp_stack_size, p.insertsize_low, p.insertsize_high = 10, 5, 80, 500
    p.max_group_size, p.max_num_junctions_to_combine = 200, 500
    p.min_subregion_overlap, p.min_guaranteed_edge_weight = 1.5, 0.01
    p.min_grouping_similarity, p.max_grouping_similarity = 0.10, 0.80
    p.min_boundary_log_ratio = 2.0
    p.max_group_boundary_distance = 10000
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def _arr(ptr, n, dtype=None):
    if n <= 0:
        return np.zeros(0, dtype or np.int32)
    return np.ctypeslib.as_array(ptr, shape=(int(n),)).copy()


class AgpuError(RuntimeError):
    """a failed ABI call; `rc` is its return code (AGPU_ERR_*)"""

    def __init__(self, msg, rc=None):
        super().__init__(msg)
        self.rc = rc


AGPU_ERR_ARG, AGPU_ERR_CUDA, AGPU_ERR_OOM, AGPU_ERR_INPUT, AGPU_ERR_CAPACITY = -1, -2, -3, -4, -5


class Context:
    """agpu_ctx: one CUDA stream.  `stream` may be a raw cudaStream_t (int), e.g. torch's current stream."""

    def __init__(self, device=0, stream=None, lib_path=None):
        self.L = load(lib_path)
        h = C.c_void_p()
        rc = self.L.agpu_create(device, C.c_void_p(stream) if stream else None, C.byref(h))
        if rc != 0:
            raise AgpuError("agpu_create(device=%d) failed with %d: no usable CUDA device (no CPU fallback)" % (device, rc))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.L.agpu_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def check(self, rc, what):
        if rc != 0:
            raise AgpuError("%s failed with %d: %s" % (what, rc, self.L.agpu_last_error(self.h).decode()), rc)

    def sync(self):
        self.check(self.L.agpu_sync(self.h), "agpu_sync")

    @property
    def launches(self):
        return self.L.agpu_launch_count(self.h)

    @property
    def syncs(self):
        """host waits on the stream so far (each one drains it)"""
        return self.L.agpu_sync_count(self.h)

    @property
    def d2h_bytes(self):
        """device -> host bytes the result fetches of this context have copied so far"""
        return self.L.agpu_d2h_bytes(self.h)

    @property
    def reserved(self):
        return self.L.agpu_reserved(self.h)

    def reserve(self, nbytes):
        self.check(self.L.agpu_reserve(self.h, int(nbytes)), "agpu_reserve")

    def pinned_match(self, other):
        """grow this context's pinned result buffers to the sizes of `other`'s (both idle)"""
        self.check(self.L.agpu_pinned_match(self.h, other.h), "agpu_pinned_match")

    def upload_async(self, on=True):
        """uploads of this context return once queued; the host buffers must outlive the batch's first stage call"""
        self.check(self.L.agpu_upload_async(self.h, 1 if on else 0), "agpu_upload_async")

    def blocking_sync(self, on=True):
        self.check(self.L.agpu_blocking_sync(self.h, 1 if on else 0), "agpu_blocking_sync")

    def profile(self, on=True):
        self.check(self.L.agpu_profile_enable(self.h, 1 if on else 0), "agpu_profile_enable")

    def profile_reset(self):
        self.check(self.L.agpu_profile_reset(self.h), "agpu_profile_reset")

    def profile_read(self):
        """{kernel: (ms, launches)} accumulated since the last reset (synchronises)"""
        buf = C.create_string_buffer(1 << 16)
        self.check(self.L.agpu_profile_read(self.h, buf, len(buf)), "agpu_profile_read")
        out = {}
        for line in buf.value.decode().splitlines():
            n, ms, cnt = line.split("\t")
            out[n] = (float(ms), int(cnt))
        return out

    def upload(self, batch_in, keepalive=None):
        """agpu_batch_upload, or agpu_batch_upload_packed when handed the compact form (hostlib.BatchPacked)"""
        return Batch(self, batch_in, False, keepalive)

    def adopt(self, batch_in_device, keepalive=None):
        return Batch(self, batch_in_device, True, keepalive)

    def gather(self, batches, picks):
        """agpu_batch_gather: a new Batch on this context whose bundle k is bundle picks[k][1] of batches[picks[k][0]], copied on the
        device.  `batches` may live on other contexts of the same device; they may be freed once this returns."""
        sel = np.asarray(picks, np.int32).reshape(-1, 2)
        src = np.ascontiguousarray(sel[:, 0])
        bun = np.ascontiguousarray(sel[:, 1])
        if any(getattr(b, "h", None) is None for b in batches):
            raise ValueError("gather: a source batch has been freed")
        tab = (C.c_void_p * max(len(batches), 1))(*[b.h.value for b in batches])
        h = C.c_void_p()
        self.check(self.L.agpu_batch_gather(self.h, len(batches), tab, len(sel), src.ctypes.data, bun.ctypes.data, C.byref(h)),
                   "agpu_batch_gather")
        return Batch.own(self, h, len(sel))

    def sort_perm(self, keys):
        keys = np.ascontiguousarray(keys, np.int32)
        perm = np.zeros(len(keys), np.int32)
        self.check(self.L.agpu_debug_sort_perm(self.h, keys.ctypes.data, len(keys), perm.ctypes.data), "agpu_debug_sort_perm")
        return perm

    def similarity(self, lists):
        """dense c (int32) and r (float64) of |A∩B| and c / min(|A|,|B|) over sorted splice lists."""
        g = len(lists)
        off = np.zeros(g + 1, np.int64)
        for i, l in enumerate(lists):
            off[i + 1] = off[i] + len(l)
        val = np.concatenate([np.asarray(l, np.int32) for l in lists]) if g and off[g] else np.zeros(0, np.int32)
        val = np.ascontiguousarray(val, np.int32)
        c = np.zeros((g, g), np.int32)
        r = np.zeros((g, g), np.float64)
        self.check(self.L.agpu_similarity(self.h, g, off.ctypes.data, val.ctypes.data, c.ctypes.data, r.ctypes.data), "agpu_similarity")
        return c, r


def _pack_lists(lists):
    g = len(lists)
    off = np.zeros(g + 1, np.int64)
    for i, l in enumerate(lists):
        off[i + 1] = off[i] + len(l)
    val = np.concatenate([np.asarray(l, np.int32) for l in lists]) if g and off[g] else np.zeros(1, np.int32)
    return off, np.ascontiguousarray(val, np.int32)


def group_resolve(ctx, lists, params):
    """bundle_group::resolve over sorted splice lists; returns the groups (lists of bundle indices) in gvv order"""
    off, val = _pack_lists(lists)
    g = len(lists)
    grp = np.zeros(max(g, 1), np.int32)
    ng = C.c_int32(0)
    ctx.check(ctx.L.agpu_group_resolve(ctx.h, g, off.ctypes.data, val.ctypes.data, C.byref(params), grp.ctypes.data, C.byref(ng)),
              "agpu_group_resolve")
    out = [[] for _ in range(ng.value)]
    for i in range(g):
        out[grp[i]].append(i)
    return out


def group_resolve_batch(ctx, groups, params):
    """bundle_group::resolve for many bundle groups in one call.  groups: list of lists of sorted splice lists.
    Returns, per bundle group, its clusters (lists of list indices local to the group) in gvv order."""
    flat = [l for grp in groups for l in grp]
    off, val = _pack_lists(flat)
    goff = np.zeros(len(groups) + 1, np.int32)
    for i, grp in enumerate(groups):
        goff[i + 1] = goff[i] + len(grp)
    out = np.zeros(max(len(flat), 1), np.int32)
    ng = np.zeros(max(len(groups), 1), np.int32)
    ctx.check(ctx.L.agpu_group_resolve_batch(ctx.h, len(groups), goff.ctypes.data, off.ctypes.data, val.ctypes.data, C.byref(params),
                                             out.ctypes.data, ng.ctypes.data), "agpu_group_resolve_batch")
    res = []
    for i, grp in enumerate(groups):
        cl = [[] for _ in range(ng[i])]
        for k in range(len(grp)):
            cl[out[goff[i] + k]].append(k)
        res.append(cl)
    return res


def group_resolve_arrays(ctx, group_off, list_off, list_val, params):
    """agpu_group_resolve_batch on packed arrays: lists ordered group by group.  Returns (cluster_of[list], n_clusters[group])."""
    group_off = np.ascontiguousarray(group_off, np.int32)
    list_off = np.ascontiguousarray(list_off, np.int64)
    list_val = np.ascontiguousarray(list_val if len(list_val) else np.zeros(1, np.int32), np.int32)
    ng = len(group_off) - 1
    out = np.zeros(max(int(group_off[-1]), 1), np.int32)
    ncl = np.zeros(max(ng, 1), np.int32)
    ctx.check(ctx.L.agpu_group_resolve_batch(ctx.h, ng, group_off.ctypes.data, list_off.ctypes.data, list_val.ctypes.data, C.byref(params),
                                             out.ctypes.data, ncl.ctypes.data), "agpu_group_resolve_batch")
    return out, ncl


def reorder_lists(off, val, order):
    """packed lists (off, val) re-packed in the order `order` (host library: one memcpy per list)"""
    from . import hostlib
    off = np.ascontiguousarray(off, np.int64)
    val = np.ascontiguousarray(val, np.int32)
    order = np.ascontiguousarray(order, np.int64)
    noff = np.zeros(len(order) + 1, np.int64)
    total = int((off[order + 1] - off[order]).sum()) if len(order) else 0
    nval = np.empty(max(total, 1), np.int32)
    got = hostlib.lib().packer_reorder_lists(len(off) - 1, off.ctypes.data, val.ctypes.data, len(order), order.ctypes.data, noff.ctypes.data, nval.ctypes.data)
    if got != total:
        raise ValueError("reorder_lists: index outside the lists")
    return noff, nval[:total]


class _DeviceArray:
    """__cuda_array_interface__ of one device column of a batch; holds the batch so that it is not collected under the tensor"""

    def __init__(self, ptr, n, typestr, owner):
        self.owner = owner
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3, "strides": None}


class Batch:
    """agpu_batch: device-resident state of a batch of bundles."""

    def __init__(self, ctx, bin_struct, adopt, keepalive):
        self.ctx = ctx
        self.keep = keepalive
        self.nb = bin_struct.n_bundles
        self.hit_off = None
        h = C.c_void_p()
        name = "agpu_batch_adopt" if adopt else ("agpu_batch_upload_packed" if hasattr(bin_struct, "hit_meta") else "agpu_batch_upload")
        ctx.check(getattr(ctx.L, name)(ctx.h, C.byref(bin_struct), C.byref(h)), name)
        self.h = h

    @classmethod
    def own(cls, ctx, handle, n_bundles):
        """a Batch around a handle an ABI call returned (e.g. agpu_batch_gather); freed with the object"""
        b = cls.__new__(cls)
        b.ctx, b.keep, b.nb, b.hit_off, b.h = ctx, None, n_bundles, None, handle
        return b

    def free(self):
        if getattr(self, "h", None) and self.ctx.h:
            self.ctx.L.agpu_batch_free(self.ctx.h, self.h)
            self.h = None

    def __del__(self):
        self.free()

    def _run(self, name, params=None):
        fn = getattr(self.ctx.L, "agpu_batch_" + name)
        rc = fn(self.ctx.h, self.h, C.byref(params)) if params is not None else fn(self.ctx.h, self.h)
        self.ctx.check(rc, "agpu_batch_" + name)

    def reset(self):
        self._run("reset")

    def evidence(self, p):
        self._run("evidence", p)

    def fragments(self):
        self._run("fragments")

    def graph(self, p):
        self._run("graph", p)

    def cluster(self, p):
        self._run("cluster", p)

    def bridge(self, p):
        self._run("bridge", p)

    def update(self):
        self._run("update")

    def bridge_all(self, p):
        self._run("bridge_all", p)

    def results(self, what=RESULT_ALL):
        """agpu_batch_results: every structure bundle::bridge leaves behind, packed on the device and copied into the context's
        pinned host buffers.  Returns the C struct of views (pointers into pinned memory, valid until the next fetch on this
        context); `.bytes` is the device -> host traffic of the call."""
        r = Results()
        self.ctx.check(self.ctx.L.agpu_batch_results(self.ctx.h, self.h, what, C.byref(r)), "agpu_batch_results")
        return r

    def counts(self):
        c = Counts()
        self.ctx.check(self.ctx.L.agpu_batch_counts(self.ctx.h, self.h, C.byref(c)), "agpu_batch_counts")
        return {n: getattr(c, n) for n, _ in Counts._fields_}

    # ---- fetches: per-bundle dicts in the oracle's array naming (tests/orclib.py) ----------
    @staticmethod
    def _chainset(v, nb, handle_off, pre, hname):
        out = []
        bco = _arr(v.bundle_chain_off, nb + 1)
        nc = int(bco[nb]) if nb else 0
        co = _arr(v.chain_off, nc + 1)
        cv = _arr(v.chain_val, int(co[nc]) if nc else 0)
        cc = _arr(v.chain_cnt, 3 * nc)
        cg = _arr(v.chain_grp, nc)
        hc = _arr(v.handle_chain, v.n_handles)
        for k in range(nb):
            a, b = int(bco[k]), int(bco[k + 1])
            o = co[a:b + 1] - (co[a] if b >= a and len(co) else 0)
            d = {pre + "_off": o.astype(np.int32), pre + "_val": cv[int(co[a]):int(co[b])], pre + "_cnt": cc[3 * a:3 * b],
                 pre + "_grp": cg[a:b]}
            if handle_off is not None:
                d[hname] = hc[int(handle_off[k]):int(handle_off[k + 1])]
            out.append(d)
        return out

    def fetch_evidence(self, hit_off):
        v = EvidenceView()
        self.ctx.check(self.ctx.L.agpu_evidence_fetch(self.ctx.h, self.h, C.byref(v)), "agpu_evidence_fetch")
        nb = self.nb
        lpos, rpos, strand = _arr(v.lpos, nb), _arr(v.rpos, nb), _arr(v.strand, nb, np.uint8)
        so = _arr(v.seg_off, nb + 1, np.int64)
        seg = _arr(v.seg, 3 * int(so[nb]) if nb else 0)
        spo = _arr(v.splice_off, nb + 1, np.int64)
        spv = _arr(v.splices, int(spo[nb]) if nb else 0)
        cs = self._chainset(v.hcst, nb, hit_off, "hcst", "hit_chain")
        out = []
        for k in range(nb):
            d = {"bundle": np.array([lpos[k], rpos[k], strand[k], hit_off[k + 1] - hit_off[k]], np.int32),
                 "seg": seg[3 * int(so[k]):3 * int(so[k + 1])], "splices": spv[int(spo[k]):int(spo[k + 1])]}
            d.update(cs[k])
            out.append(d)
        return out

    def phase_set(self):
        """bundle_base::build_phase_set against the current graphs; per bundle the oracle's phase_off / phase_val / phase_cnt"""
        self._run("phase_set")
        v = PhaseView()
        self.ctx.check(self.ctx.L.agpu_phase_fetch(self.ctx.h, self.h, C.byref(v)), "agpu_phase_fetch")
        nb, npz = self.nb, int(v.n_phases)
        po = _arr(v.phase_off, nb + 1, np.int64)
        co = _arr(v.coord_off, npz + 1, np.int64)
        cv = _arr(v.coords, int(co[npz]) if npz else 0)
        cc = _arr(v.count, npz)
        out = []
        for k in range(nb):
            a, b = int(po[k]), int(po[k + 1])
            out.append({"phase_off": (co[a:b + 1] - co[a]).astype(np.int32), "phase_val": cv[int(co[a]):int(co[b])], "phase_cnt": cc[a:b]})
        return out

    def raw_views(self):
        """the C structs of agpu_graph_fetch / agpu_revise_fetch / agpu_phase_fetch as a foreign caller sees them (pointers
        stay valid until the next fetch of the same kind); the stages must have run"""
        g, r, p = GraphView(), ReviseView(), PhaseView()
        self.ctx.check(self.ctx.L.agpu_graph_fetch(self.ctx.h, self.h, C.byref(g)), "agpu_graph_fetch")
        self.ctx.check(self.ctx.L.agpu_revise_fetch(self.ctx.h, self.h, C.byref(r)), "agpu_revise_fetch")
        self.ctx.check(self.ctx.L.agpu_phase_fetch(self.ctx.h, self.h, C.byref(p)), "agpu_phase_fetch")
        return g, r, p

    def revise(self, p, fetch=True):
        """identify_boundaries + remove_false_boundaries on the bundles' graphs; per bundle the oracle's rev_edge / rev_edge_d /
        rev_vert / rev_vert_d"""
        self._run("revise", p)
        if not fetch:
            return None
        v = ReviseView()
        self.ctx.check(self.ctx.L.agpu_revise_fetch(self.ctx.h, self.h, C.byref(v)), "agpu_revise_fetch")
        nb, ne, nv = self.nb, int(v.n_edges), int(v.n_vertices)
        eo, vo = _arr(v.edge_off, nb + 1, np.int64), _arr(v.vert_off, nb + 1, np.int64)
        e, ew = _arr(v.edge, 2 * ne), _arr(v.edge_w, ne, np.float64)
        c, r = _arr(v.unbridge, 2 * nv), _arr(v.unbridge_ratio, 2 * nv, np.float64)
        out = []
        for k in range(nb):
            a, b, x, y = int(eo[k]), int(eo[k + 1]), int(vo[k]), int(vo[k + 1])
            out.append({"rev_edge": e[2 * a:2 * b], "rev_edge_d": ew[a:b], "rev_vert": c[2 * x:2 * y], "rev_vert_d": r[2 * x:2 * y]})
        return out

    def group_bridge(self, groups, p):
        """assembler::bridge over clusters of bundles: groups = list of lists of bundle indices (the reference's gv order)"""
        off = np.zeros(len(groups) + 1, np.int32)
        for i, grp in enumerate(groups):
            off[i + 1] = off[i] + len(grp)
        mem = np.ascontiguousarray(np.concatenate([np.asarray(x, np.int32) for x in groups]) if groups else np.zeros(1, np.int32), np.int32)
        self._groups = [list(map(int, x)) for x in groups]
        self.ctx.check(self.ctx.L.agpu_batch_group_bridge(self.ctx.h, self.h, len(groups), off.ctypes.data, mem.ctypes.data, C.byref(p)),
                       "agpu_batch_group_bridge")

    def coverage_edit(self, skip=None, extra=None):
        """agpu_batch_coverage_edit (insert-size preview): per-hit masks of the BAM_CMATCH blocks without coverage, extra intervals"""
        sk = np.ascontiguousarray(skip, np.uint16) if skip is not None else None
        ex = [np.ascontiguousarray(x, np.int32) for x in extra] if extra is not None and len(extra[0]) else None
        self.ctx.check(self.ctx.L.agpu_batch_coverage_edit(self.ctx.h, self.h, sk.ctypes.data if sk is not None and len(sk) else None,
                                                           len(ex[0]) if ex else 0, *([x.ctypes.data for x in ex] if ex else [None] * 4)),
                       "agpu_batch_coverage_edit")

    def preview(self, p):
        """previewer::process for every bundle: (clu_off[NB + 1], isize[C]) -- the fragment length the previewer enters into its
        histogram per paired-read cluster, INT32_MIN where it enters none"""
        self._run("preview", p)
        v = PreviewView()
        self.ctx.check(self.ctx.L.agpu_preview_fetch(self.ctx.h, self.h, C.byref(v)), "agpu_preview_fetch")
        return _arr(v.clu_off, self.nb + 1, np.int64), _arr(v.isize, int(v.n_clusters))

    def group_support(self, groups, p, fetch=True):
        """the cross-sample support features of assembler::assemble(vector<bundle*>) over clusters of bundles (lists of bundle
        indices in the reference's gv order).  Returns, per cluster, a dict in the oracle's naming (tests/orclib.py): m<k>_sup_* for
        member k, x_sup_* for the combined graph."""
        off = np.zeros(len(groups) + 1, np.int32)
        for i, grp in enumerate(groups):
            off[i + 1] = off[i] + len(grp)
        mem = np.ascontiguousarray(np.concatenate([np.asarray(x, np.int32) for x in groups]) if groups else np.zeros(1, np.int32), np.int32)
        self.ctx.check(self.ctx.L.agpu_batch_group_support(self.ctx.h, self.h, len(groups), off.ctypes.data, mem.ctypes.data, C.byref(p)),
                       "agpu_batch_group_support")
        if not fetch:
            return None
        v = SupportView()
        self.ctx.check(self.ctx.L.agpu_support_fetch(self.ctx.h, self.h, C.byref(v)), "agpu_support_fetch")
        G = int(v.n_graphs)
        vo, eo = _arr(v.vert_off, G + 1, np.int64), _arr(v.edge_off, G + 1, np.int64)
        V, E = (int(vo[G]), int(eo[G])) if G else (0, 0)
        loss, edge, abd = _arr(v.loss, 4 * V, np.float64), _arr(v.edge, 3 * E), _arr(v.abd, E, np.float64)
        so = _arr(v.sample_off, E + 1, np.int64)
        nnz = int(so[E]) if E else 0
        smp, sabd = _arr(v.sample, nnz), _arr(v.sample_abd, nnz, np.float64)
        nm = int(off[-1])

        def rows(g, pre):
            a, b, x, y = int(eo[g]), int(eo[g + 1]), int(vo[g]), int(vo[g + 1])
            r0, r1 = (int(so[a]), int(so[b])) if b > a else (0, 0)
            return {pre + "sup_edge": edge[3 * a:3 * b], pre + "sup_abd": abd[a:b], pre + "sup_loss": loss[4 * x:4 * y],
                    pre + "sup_off": (so[a:b + 1] - so[a]).astype(np.int32), pre + "sup_sample": smp[r0:r1], pre + "sup_sabd": sabd[r0:r1],
                    pre + "sup_set_off": (so[a:b + 1] - so[a]).astype(np.int32), pre + "sup_set": smp[r0:r1]}
        out = []
        for i, grp in enumerate(groups):
            d = {}
            for k in range(len(grp)):
                d.update(rows(int(off[i]) + k, "m%d_" % k))
            d.update(rows(nm + i, "x_"))
            out.append(d)
        return out

    def fetch_group(self):
        """per cluster of the last group_bridge: dict with the oracle's cb_* arrays (tests/orclib.py naming) + combine_order"""
        ev, fc, gv, po = EvidenceView(), ChainsetView(), GraphView(), P32()
        self.ctx.check(self.ctx.L.agpu_group_fetch(self.ctx.h, self.h, C.byref(ev), C.byref(fc), C.byref(gv), C.byref(po)), "agpu_group_fetch")
        ng = len(self._groups)
        nmem = sum(len(x) for x in self._groups)
        order = _arr(po, nmem)
        lpos, rpos, strand = _arr(ev.lpos, ng), _arr(ev.rpos, ng), _arr(ev.strand, ng, np.uint8)
        so = _arr(ev.seg_off, ng + 1, np.int64)
        seg = _arr(ev.seg, 3 * int(so[ng]) if ng else 0)
        hc = self._chainset(ev.hcst, ng, None, "cb_hcst", None)
        fcs = self._chainset(fc, ng, None, "cb_fcst", None)
        jo, pox, vo, eo = (_arr(x, ng + 1) for x in (gv.junc_off, gv.pexon_off, gv.vert_off, gv.edge_off))
        junc, pex, vert, edge = _arr(gv.junc, 9 * int(jo[ng])), _arr(gv.pexon, 5 * int(pox[ng])), _arr(gv.vert, 5 * int(vo[ng])), _arr(gv.edge, 3 * int(eo[ng]))
        pexd, vertd, edged = _arr(gv.pexon_d, 4 * int(pox[ng]), np.float64), _arr(gv.vert_d, 3 * int(vo[ng]), np.float64), _arr(gv.edge_d, int(eo[ng]), np.float64)
        out = []
        m0 = 0
        for k in range(ng):
            n = len(self._groups[k])
            d = {"combine_order": np.array([self._groups[k].index(int(m)) for m in order[m0:m0 + n]], np.int32),
                 "cb_bundle": np.array([lpos[k], rpos[k], strand[k]], np.int32), "cb_seg": seg[3 * int(so[k]):3 * int(so[k + 1])],
                 "cb_junc": junc[9 * int(jo[k]):9 * int(jo[k + 1])], "cb_pexon": pex[5 * int(pox[k]):5 * int(pox[k + 1])],
                 "cb_pexon_d": pexd[4 * int(pox[k]):4 * int(pox[k + 1])], "cb_vert": vert[5 * int(vo[k]):5 * int(vo[k + 1])],
                 "cb_vert_d": vertd[3 * int(vo[k]):3 * int(vo[k + 1])]}
            e = edge[3 * int(eo[k]):3 * int(eo[k + 1])].reshape(-1, 3)
            ew = edged[int(eo[k]):int(eo[k + 1])]
            alive = e[:, 0] >= 0
            ea, wa = e[alive], ew[alive]
            o2 = np.lexsort((ea[:, 1], ea[:, 0])) if len(ea) else np.zeros(0, np.int64)
            d["cb_edge"] = ea[o2].reshape(-1).astype(np.int32)
            d["cb_edge_d"] = wa[o2]
            d.update(hc[k])
            d.update(fcs[k])
            out.append(d)
            m0 += n
        return out

    INPUT_COLUMNS = [("bundle_hit_off", "nb1", "<i8"), ("pos", "nh", "<i4"), ("rpos", "nh", "<i4"), ("mpos", "nh", "<i4"),
                     ("isize", "nh", "<i4"), ("strand", "nh", "|i1"), ("bundle_strand", "nb", "|i1"), ("xs", "nh", "|i1"),
                     ("qid", "nh", "<i8"), ("cigar_off", "nh1", "<i4"), ("cigar", "nc", "<i4")]

    def input_columns(self):
        """agpu_batch_inputs: the input columns the stages read, as zero-copy torch tensors over the batch's device arrays (CPU
        tensors over host memory on the emulation build), unsigned columns viewed as signed ones of the same width.  Of strand and
        bundle_strand only the one the batch has is present.  Valid until the batch is freed; no stage writes them."""
        import torch
        v = BatchIn()
        self.ctx.check(self.ctx.L.agpu_batch_inputs(self.ctx.h, self.h, C.byref(v)), "agpu_batch_inputs")
        size = {"nb": v.n_bundles, "nb1": v.n_bundles + 1, "nh": v.n_hits, "nh1": v.n_hits + 1, "nc": v.n_cigar}
        out = {}
        for name, n, typestr in self.INPUT_COLUMNS:
            ptr, n = getattr(v, name), int(size[n])
            if not ptr:
                continue
            dt = np.dtype(typestr)
            if n == 0:
                out[name] = torch.empty(0, dtype=torch.from_numpy(np.zeros(0, dt)).dtype)
            elif self.ctx.L.host_memory:
                out[name] = torch.from_numpy(np.ctypeslib.as_array(C.cast(ptr, C.POINTER(np.ctypeslib.as_ctypes_type(dt))), shape=(n,)))
            else:
                out[name] = torch.as_tensor(_DeviceArray(ptr, n, typestr, self), device="cuda")
        return out

    def bundle_counts(self):
        """[NB, 4] int64: segments, fragments, clusters, bridged pairs of every bundle"""
        out = np.zeros((max(self.nb, 1), 4), np.int64)
        self.ctx.check(self.ctx.L.agpu_batch_bundle_counts(self.ctx.h, self.h, out.ctypes.data), "agpu_batch_bundle_counts")
        return out[:self.nb]

    def fetch_splices(self):
        """(splice_off[NB+1], splices) as numpy arrays: bundle::splices of every bundle"""
        po, pv = P64(), P32()
        self.ctx.check(self.ctx.L.agpu_splices_fetch(self.ctx.h, self.h, C.byref(po), C.byref(pv)), "agpu_splices_fetch")
        off = _arr(po, self.nb + 1, np.int64)
        return off, _arr(pv, int(off[self.nb]) if self.nb else 0)

    def fetch_graph(self):
        v = GraphView()
        self.ctx.check(self.ctx.L.agpu_graph_fetch(self.ctx.h, self.h, C.byref(v)), "agpu_graph_fetch")
        nb = self.nb
        jo, po, vo, eo = (_arr(x, nb + 1) for x in (v.junc_off, v.pexon_off, v.vert_off, v.edge_off))
        junc, pex, vert, edge = _arr(v.junc, 9 * int(jo[nb])), _arr(v.pexon, 5 * int(po[nb])), _arr(v.vert, 5 * int(vo[nb])), _arr(v.edge, 3 * int(eo[nb]))
        pexd, vertd, edged = _arr(v.pexon_d, 4 * int(po[nb]), np.float64), _arr(v.vert_d, 3 * int(vo[nb]), np.float64), _arr(v.edge_d, int(eo[nb]), np.float64)
        strand = _arr(v.strand, nb, np.uint8)
        out = []
        for k in range(nb):
            e = edge[3 * int(eo[k]):3 * int(eo[k + 1])].reshape(-1, 3)
            ew = edged[int(eo[k]):int(eo[k + 1])]
            alive = e[:, 0] >= 0
            out.append({"junc": junc[9 * int(jo[k]):9 * int(jo[k + 1])], "pexon": pex[5 * int(po[k]):5 * int(po[k + 1])],
                        "pexon_d": pexd[4 * int(po[k]):4 * int(po[k + 1])], "vert": vert[5 * int(vo[k]):5 * int(vo[k + 1])],
                        "vert_d": vertd[3 * int(vo[k]):3 * int(vo[k + 1])],
                        "edge_ins": e[alive].reshape(-1), "edge_ins_d": ew[alive],     # insertion order, alive only
                        "graph": np.array([strand[k]], np.int32)})
            # oracle convention: edges sorted by (s, t)
            ea, wa = e[alive], ew[alive]
            order = np.lexsort((ea[:, 1], ea[:, 0])) if len(ea) else np.zeros(0, np.int64)
            out[-1]["edge"] = ea[order].reshape(-1).astype(np.int32)
            out[-1]["edge_d"] = wa[order]
        return out

    def fetch_fragments(self):
        v = FragmentsView()
        self.ctx.check(self.ctx.L.agpu_fragments_fetch(self.ctx.h, self.h, C.byref(v)), "agpu_fragments_fetch")
        nb = self.nb
        fo = _arr(v.frg_off, nb + 1, np.int64)
        fr = _arr(v.frgs, 3 * int(fo[nb]) if nb else 0)
        br = _arr(v.bridged, nb)
        cs = self._chainset(v.fcst, nb, fo, "fcst", "frg_chain")
        out = []
        for k in range(nb):
            d = {"frgs": fr[3 * int(fo[k]):3 * int(fo[k + 1])], "bridged": br[k:k + 1]}
            d.update(cs[k])
            out.append(d)
        return out

    def fetch_clusters(self, evidence):
        """`evidence`: result of fetch_evidence (chain indices are expanded to coordinates)."""
        v = ClusterView()
        self.ctx.check(self.ctx.L.agpu_cluster_fetch(self.ctx.h, self.h, C.byref(v)), "agpu_cluster_fetch")
        nb = self.nb
        co = _arr(v.clu_off, nb + 1, np.int64)
        nc = int(v.n_clusters)
        bo, ex, ct = _arr(v.bounds, 4 * nc), _arr(v.extend, 4 * nc), _arr(v.count, nc)
        c1, c2 = _arr(v.chain1, nc), _arr(v.chain2, nc)
        fo = _arr(v.frlist_off, nc + 1, np.int64)
        fl = _arr(v.frlist, int(fo[nc]) if nc else 0)
        out = []
        for k in range(nb):
            a, b = int(co[k]), int(co[k + 1])
            ev = evidence[k]

            def chains(idx):
                off, val = [0], []
                for c in idx:
                    if c >= 0:
                        val.extend(ev["hcst_val"][ev["hcst_off"][c]:ev["hcst_off"][c + 1]].tolist())
                    off.append(len(val))
                return np.array(off, np.int32), np.array(val, np.int32)
            o1, v1 = chains(c1[a:b])
            o2, v2 = chains(c2[a:b])
            out.append({"clu_bounds": bo[4 * a:4 * b], "clu_extend": ex[4 * a:4 * b], "clu_count": ct[a:b],
                        "clu_c1_off": o1, "clu_c1_val": v1, "clu_c2_off": o2, "clu_c2_val": v2,
                        "clu_fr_off": (fo[a:b + 1] - fo[a]).astype(np.int32), "clu_fr_val": fl[int(fo[a]):int(fo[b])]})
        return out

    def fetch_bridge(self, clu_off):
        v = BridgeView()
        self.ctx.check(self.ctx.L.agpu_bridge_fetch(self.ctx.h, self.h, C.byref(v)), "agpu_bridge_fetch")
        nb = self.nb
        nc = int(clu_off[nb]) if nb else 0
        ty, st, ch = _arr(v.type, nc), _arr(v.strand, nc), _arr(v.choices, nc)
        sc = _arr(v.score, nc, np.float64)
        co, wo = _arr(v.chain_off, nc + 1, np.int64), _arr(v.whole_off, nc + 1, np.int64)
        cv, wv = _arr(v.chain, int(co[nc]) if nc else 0), _arr(v.whole, int(wo[nc]) if nc else 0)
        out = []
        for k in range(nb):
            a, b = int(clu_off[k]), int(clu_off[k + 1])
            opt = np.stack([ty[a:b], st[a:b], ch[a:b]], axis=1).reshape(-1).astype(np.int32) if b > a else np.zeros(0, np.int32)
            out.append({"opt": opt, "opt_score": sc[a:b],
                        "opt_chain_off": (co[a:b + 1] - co[a]).astype(np.int32), "opt_chain_val": cv[int(co[a]):int(co[b])],
                        "opt_whole_off": (wo[a:b + 1] - wo[a]).astype(np.int32), "opt_whole_val": wv[int(wo[a]):int(wo[b])]})
        return out

    def cluster_offsets(self):
        v = ClusterView()
        self.ctx.check(self.ctx.L.agpu_cluster_fetch(self.ctx.h, self.h, C.byref(v)), "agpu_cluster_fetch")
        return _arr(v.clu_off, self.nb + 1, np.int64)
