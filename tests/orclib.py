"""ctypes bindings of the two CPU checkers (oracle/orc_api.h).  TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libaletsch_ref.so")
ORC_SO = os.path.join(ROOT, "oracle", "liboracle.so")


class BundleIn(C.Structure):
    _fields_ = [("n_hits", C.c_int32), ("tid", C.c_int32), ("pos", C.c_void_p), ("mpos", C.c_void_p), ("isize", C.c_void_p),
                ("flag", C.c_void_p), ("strand", C.c_void_p), ("xs", C.c_void_p), ("qid", C.c_void_p),
                ("cigar_off", C.c_void_p), ("cigar", C.c_void_p)]


class Params(C.Structure):
    """orc_params == agpu_params field for field."""
    _fields_ = [("library_type", C.c_int32), ("min_junction_support", C.c_int32), ("normal_junction_threshold", C.c_int32),
                ("extend_junction_threshold", C.c_int32), ("min_subregion_gap", C.c_int32), ("min_subregion_length", C.c_int32),
                ("max_reads_partition_gap", C.c_int32), ("bridge_end_relaxing", C.c_int32),
                ("bridge_dp_solution_size", C.c_int32), ("bridge_dp_stack_size", C.c_int32), ("insertsize_low", C.c_int32),
                ("insertsize_high", C.c_int32), ("max_group_size", C.c_int32), ("max_num_junctions_to_combine", C.c_int32),
                ("min_subregion_overlap", C.c_double), ("min_guaranteed_edge_weight", C.c_double),
                ("min_grouping_similarity", C.c_double), ("max_grouping_similarity", C.c_double),
                ("min_boundary_log_ratio", C.c_double), ("max_group_boundary_distance", C.c_int32)]


def default_params(**kw):
    """defaults of util/parameters.cc:19-113 and rnacore/sample_profile.cc:17-33."""
    p = Params(library_type=1, min_junction_support=1, normal_junction_threshold=10, extend_junction_threshold=20,
               min_subregion_gap=15, min_subregion_length=15, max_reads_partition_gap=10, bridge_end_relaxing=10,
               bridge_dp_solution_size=10, bridge_dp_stack_size=5, insertsize_low=80, insertsize_high=500,
               max_group_size=200, max_num_junctions_to_combine=500, min_subregion_overlap=1.5,
               min_guaranteed_edge_weight=0.01, min_grouping_similarity=0.10, max_grouping_similarity=0.80, min_boundary_log_ratio=2.0,
               max_group_boundary_distance=10000)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


class Checker:
    """one of the CPU checkers: prefix 'ref' (reference TUs) or 'orc' (restatement)."""

    def __init__(self, prefix):
        self.prefix = prefix
        path = REF_SO if prefix == "ref" else ORC_SO
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.lib = L = C.CDLL(path)
        L.orc_bag_new.restype = C.c_void_p
        L.orc_bag_free.argtypes = [C.c_void_p]
        L.orc_bag_clear.argtypes = [C.c_void_p]
        L.orc_bag_count.argtypes = [C.c_void_p]
        L.orc_bag_name.restype = C.c_char_p
        L.orc_bag_name.argtypes = [C.c_void_p, C.c_int]
        L.orc_bag_kind.argtypes = [C.c_void_p, C.c_int]
        L.orc_bag_len.restype = C.c_int64
        L.orc_bag_len.argtypes = [C.c_void_p, C.c_int]
        L.orc_bag_data.restype = C.c_void_p
        L.orc_bag_data.argtypes = [C.c_void_p, C.c_int]
        f = lambda n: getattr(L, prefix + "_" + n)
        f("bundle_new").restype = C.c_void_p
        f("bundle_new").argtypes = [C.POINTER(BundleIn), C.POINTER(Params)]
        f("bundle_free").argtypes = [C.c_void_p]
        for n in ("bundle_evidence", "bundle_fragments", "bundle_graph", "bundle_bridge", "bundle_phase", "bundle_revise"):
            f(n).argtypes = [C.c_void_p, C.c_void_p]
        f("group_bridge").argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_void_p]
        f("group_resolve").argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(Params), C.c_void_p]
        self.f = f

    def bag_to_dict(self, bag):
        L = self.lib
        out = {}
        for i in range(L.orc_bag_count(bag)):
            name = L.orc_bag_name(bag, i).decode()
            kind = L.orc_bag_kind(bag, i)
            n = L.orc_bag_len(bag, i)
            dt = np.int32 if kind == 0 else np.float64
            if n == 0:
                out[name] = np.zeros(0, dt)
            else:
                ct = C.c_int32 if kind == 0 else C.c_double
                out[name] = np.ctypeslib.as_array(C.cast(L.orc_bag_data(bag, i), C.POINTER(ct)), shape=(n,)).copy()
        return out

    def new_bundle(self, bd, params):
        """bd: dict of arrays of ONE bundle (PackedBatch.bundle(k))."""
        b = BundleIn()
        b.n_hits = len(bd["pos"])
        b.tid = bd["tid"]
        keep = []
        for k in ("pos", "mpos", "isize", "flag", "strand", "xs", "qid", "cigar_off", "cigar"):
            arr = np.ascontiguousarray(bd[k])
            keep.append(arr)
            setattr(b, k, arr.ctypes.data)
        h = self.f("bundle_new")(C.byref(b), C.byref(params))
        return h

    def free_bundle(self, h):
        self.f("bundle_free")(h)

    def run(self, h, stage):
        """stage in evidence / fragments / graph / bridge; returns (rc, dict)."""
        bag = self.lib.orc_bag_new()
        rc = self.f("bundle_" + stage)(h, bag)
        d = self.bag_to_dict(bag)
        self.lib.orc_bag_free(bag)
        return rc, d

    def run_quiet(self, h, stage):
        """run a stage for timing: the result bag is filled by the checker but not copied out"""
        bag = self.lib.orc_bag_new()
        rc = self.f("bundle_" + stage)(h, bag)
        self.lib.orc_bag_free(bag)
        return rc

    def group_bridge(self, hs):
        bag = self.lib.orc_bag_new()
        arr = (C.c_void_p * len(hs))(*hs)
        rc = self.f("group_bridge")(arr, len(hs), bag)
        d = self.bag_to_dict(bag)
        self.lib.orc_bag_free(bag)
        return rc, d

    def group_resolve(self, hs, params):
        bag = self.lib.orc_bag_new()
        arr = (C.c_void_p * len(hs))(*hs)
        rc = self.f("group_resolve")(arr, len(hs), C.byref(params), bag)
        d = self.bag_to_dict(bag)
        self.lib.orc_bag_free(bag)
        return rc, d
