"""ctypes binding of libogb.so (include/ogb.h). There is no fallback: a missing library raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OGB_LIB") or os.path.join(_HERE, "libogb.so")   # OGB_LIB: another build of the same library (experiments)

OGB_OK, OGB_E_ARG, OGB_E_CUDA, OGB_E_NCCL, OGB_E_STATE, OGB_E_CAPACITY, OGB_E_IO, OGB_E_NOMEM = range(8)


class OgbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libogb error {code}: {msg}")
        self.code = code


class Edge(C.Structure):
    """ogb_edge (include/ogb.h) = flat form of the reference Edge record (Edge.h:17-44)."""
    _fields_ = [("src", C.c_uint32), ("dst", C.c_uint32), ("offset", C.c_uint16), ("orient", C.c_uint8),
                ("reserved", C.c_uint8)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "n_reads", "table_buckets", "table_bytes", "n_contained", "contain_probes", "contain_hits",
        "overlap_probes", "probe_sectors", "candidates", "edges_pre", "edges_pre_local", "pivot_entries",
        "active_pivots", "edges_final", "nodes_final", "max_degree", "overflow_reads")] + [
        ("kernel_launches", C.c_uint32), ("probe_launches", C.c_uint32), ("hash_partitions", C.c_uint32), ("hash_build_attempts", C.c_uint32)] + [(n, C.c_float) for n in (
            "ms_pack", "ms_hash_build", "ms_contain", "ms_overlap", "ms_exchange_pre", "ms_mark", "ms_reduce",
            "ms_total", "ms_scan_kernel", "ms_probe_launch", "ms_window_launch")] + [
        ("ms_kernel", C.c_float * 20), ("n_kernel", C.c_uint32 * 20)]

    KERNEL_CLASSES = ("hash_insert", "window_part", "probe_parts", "verify", "rows_finish", "mark_fast1", "mark_fast2", "mark_any", "keep", "emit",
                      "contain_window", "contain_probe", "contain_verify", "exch_index", "exch_rows", "exch_bits", "exch_final", "probe_verify")

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if n not in ("ms_kernel", "n_kernel")}
        d["kernels"] = {k: {"ms": float(self.ms_kernel[i]), "launches": int(self.n_kernel[i])} for i, k in enumerate(self.KERNEL_CLASSES) if self.n_kernel[i]}
        return d


class SimplifyStats(C.Structure):
    """ogb_simplify_stats (include/ogb.h)."""
    _fields_ = [(n, C.c_uint64) for n in ("n_edges_in", "n_edges_out", "n_items", "merges", "dead_ends")] + [
        (n, C.c_uint32) for n in ("iterations", "rounds", "jumps", "launches")] + [
        (n, C.c_float) for n in ("ms", "ms_setup", "ms_sweeps", "ms_dead_ends", "ms_lists")] + [("reserved", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved"}


class SpellStats(C.Structure):
    """ogb_spell_stats (include/ogb.h)."""
    _fields_ = [(n, C.c_uint64) for n in ("unitigs", "bases", "words")] + [("launches", C.c_uint32), ("ms", C.c_float)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class CoverageStats(C.Structure):
    """ogb_coverage_stats (include/ogb.h)."""
    _fields_ = [(n, C.c_uint64) for n in ("unitigs", "bases", "placements", "contained_placements", "unplaced")] + [("launches", C.c_uint32)] + [
        (n, C.c_float) for n in ("ms", "ms_locate", "ms_depth", "ms_reduce")] + [("reserved", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved"}


class MapStats(C.Structure):
    """ogb_map_stats (include/ogb.h)."""
    _fields_ = [(n, C.c_uint64) for n in ("reads_in", "filtered", "mapped", "multi", "placements", "index_entries", "index_buckets")] + [
        (n, C.c_uint32) for n in ("sample", "launches")] + [(n, C.c_float) for n in ("ms", "ms_index", "ms_upload", "ms_map", "ms_reduce")] + [
        ("reserved", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved"}


OGB_MAP_FILTERED = 0xFFFFFFFF
OGB_MAP_UNPLACED = 0xFF
OGB_MAP_MAX_MISMATCHES = 8

# every symbol include/ogb.h declares: name -> (restype, argtypes)
_u64p = C.POINTER(C.c_uint64)
_vp = C.c_void_p
PROTOTYPES = {
    "ogb_version": (C.c_int, []),
    "ogb_last_error": (C.c_char_p, []),
    "ogb_dataset_create": (C.c_int, [C.POINTER(_vp)]),
    "ogb_dataset_destroy": (None, [_vp]),
    "ogb_dataset_add_reads": (C.c_int, [_vp, _vp, _vp, C.c_uint64]),
    "ogb_dataset_add_file": (C.c_int, [_vp, C.c_char_p]),
    "ogb_dataset_finalize": (C.c_int, [_vp, C.c_uint32]),
    "ogb_dataset_finalize_device": (C.c_int, [_vp, _vp, C.c_uint32]),
    "ogb_dataset_n_reads": (C.c_uint64, [_vp]),
    "ogb_dataset_n_unique": (C.c_uint64, [_vp]),
    "ogb_dataset_shortest": (C.c_uint64, [_vp]),
    "ogb_dataset_longest": (C.c_uint64, [_vp]),
    "ogb_dataset_min_overlap": (C.c_uint32, [_vp]),
    "ogb_dataset_words": (_vp, [_vp, _u64p]),
    "ogb_dataset_word_offsets": (_vp, [_vp]),
    "ogb_dataset_lengths": (_vp, [_vp]),
    "ogb_dataset_frequencies": (_vp, [_vp]),
    "ogb_dataset_get_read": (C.c_int, [_vp, C.c_uint64, C.c_int, _vp, C.c_uint32, C.POINTER(C.c_uint32)]),
    "ogb_dataset_find_read": (C.c_int, [_vp, C.c_char_p, C.c_uint32, _u64p]),
    "ogb_dataset_raw_reads": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), _u64p]),
    "ogb_context_create": (C.c_int, [C.POINTER(_vp), C.c_int]),
    "ogb_nccl_unique_id": (C.c_int, [_vp]),
    "ogb_context_create_dist": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int, C.c_int, _vp]),
    "ogb_context_destroy": (None, [_vp]),
    "ogb_context_rank": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ogb_reads_upload": (C.c_int, [_vp, _vp, _vp, C.c_uint64]),
    "ogb_reads_upload_packed": (C.c_int, [_vp, _vp, _vp, _vp, C.c_uint64]),
    "ogb_reads_upload_dataset": (C.c_int, [_vp, _vp]),
    "ogb_reads_upload_packed_sharded": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint32]),
    "ogb_hash_build": (C.c_int, [_vp, C.c_uint32]),
    "ogb_hash_lookup": (C.c_int, [_vp, _vp, C.c_uint64, _vp, C.c_uint64, _vp]),
    "ogb_hash_string_length": (C.c_uint64, [_vp]),
    "ogb_hash_table_size": (C.c_uint64, [_vp]),
    "ogb_mark_contained": (C.c_int, [_vp]),
    "ogb_super_read_ids": (C.c_int, [_vp, _vp, C.c_uint64]),
    "ogb_mate_lookup": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_uint32, _vp, _vp]),
    "ogb_build_graph": (C.c_int, [_vp, C.c_int]),
    "ogb_graph_edge_count": (C.c_int, [_vp, C.c_int, _u64p]),
    "ogb_graph_edges": (C.c_int, [_vp, C.c_int, _vp, C.c_uint64]),
    "ogb_graph_edges_shard": (C.c_int, [_vp, _vp, C.c_uint64, _u64p]),
    "ogb_graph_checksum": (C.c_int, [_vp, C.c_int, _u64p, _u64p]),
    "ogb_graph_simplify": (C.c_int, [_vp, C.POINTER(SimplifyStats)]),
    "ogb_graph_composite_edges": (C.c_int, [_vp, _vp, C.c_uint64, _vp, C.c_uint64]),
    "ogb_graph_spell": (C.c_int, [_vp, C.c_int, C.c_uint64, C.c_uint64, C.POINTER(SpellStats)]),
    "ogb_graph_unitigs": (C.c_int, [_vp, _vp, C.c_uint64, _vp, C.c_uint64, C.c_int]),
    "ogb_graph_write_unitigs": (C.c_int, [_vp, C.c_char_p]),
    "ogb_graph_coverage": (C.c_int, [_vp, _vp, C.c_uint64, C.POINTER(CoverageStats)]),
    "ogb_graph_unitig_coverage": (C.c_int, [_vp, _vp, C.c_uint64, _vp, C.c_uint64]),
    "ogb_graph_write_coverage": (C.c_int, [_vp, C.c_char_p]),
    "ogb_graph_map_reads": (C.c_int, [_vp, _vp, _vp, C.c_uint64, _vp, C.POINTER(MapStats)]),
    "ogb_graph_map_reads_approx": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_uint32, _vp, _vp, C.POINTER(MapStats)]),
    "ogb_graph_sample_coverage": (C.c_int, [_vp, C.c_uint32, _vp, C.c_uint64, _vp, C.c_uint64]),
    "ogb_graph_write_depths": (C.c_int, [_vp, C.c_char_p, _vp]),
    "ogb_get_stats": (C.c_int, [_vp, C.POINTER(Stats)]),
    "ogb_timer_begin": (C.c_int, [_vp]),
    "ogb_timer_end": (C.c_int, [_vp, C.POINTER(C.c_float)]),
    "ogb_l2_flush": (C.c_int, [_vp, C.c_size_t]),
    "ogb_gather_ceiling": (C.c_int, [_vp, C.c_size_t, C.c_uint32, C.POINTER(C.c_double)]),
    "ogb_alloc_host": (C.c_int, [C.POINTER(_vp), C.c_size_t]),
    "ogb_free_host": (None, [_vp]),
    "ogb_synth_genome": (C.c_int, [C.c_uint64, C.c_uint64, _vp]),
    "ogb_synth_reads": (C.c_int, [C.c_uint64, _vp, _vp, _vp, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int,
                                  C.c_double, C.c_double, _vp, C.c_uint64, _vp]),
}

_lib = None


def lib():
    """Loads libogb.so (built in-tree by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OgbError(-1, f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)")
        l = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in PROTOTYPES.items():
            f = getattr(l, name)  # AttributeError if the library does not export a declared symbol
            f.restype, f.argtypes = res, args
        _lib = l
    return _lib


def check(rc):
    if rc != OGB_OK:
        raise OgbError(rc, lib().ogb_last_error().decode("utf-8", "replace"))
