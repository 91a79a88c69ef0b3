"""Python mirror of the reference's call-site classes over the libogb C ABI.

The product host API is the C++ one in metagenomics_b200/host/ (same class names and signatures as
MetaGenomics/{Dataset,HashTable,OverlapGraph,Edge}.h). This module mirrors the same three steps --
``Dataset(...)``, ``HashTable().insertDataset(ds, minOverlap)``, ``OverlapGraph(hashTable)``
(MetaGenomics/main.cpp:33,45-47) -- for bench.py and the parity tests, calling the very same C entry
points. Nothing here computes on the CPU; without a GPU the device calls raise OgbError.
"""
import ctypes as C

import numpy as np

from ._lib import Edge, OgbError, Stats, check, lib  # noqa: F401

EDGE_DTYPE = np.dtype([("src", "<u4"), ("dst", "<u4"), ("offset", "<u2"), ("orient", "u1"), ("reserved", "u1")])
# ogb_cedge / ogb_clist_item (include/ogb.h): the simplified graph
CEDGE_DTYPE = np.dtype([("src", "<u4"), ("dst", "<u4"), ("offset", "<u8"), ("list_start", "<u8"), ("count", "<u4"), ("twin", "<u4"), ("orient", "u1"),
                        ("reserved", "u1", (3,)), ("reserved2", "<u4")])
CITEM_DTYPE = np.dtype([("read", "<u4"), ("offset", "<u2"), ("orient", "u1"), ("reserved", "u1")])
# ogb_unitig: one spelled unitig; its sequence is bases [start, start + length) of the word-aligned layout (OverlapGraph.unitigs)
UNITIG_DTYPE = np.dtype([("edge", "<u4"), ("src", "<u4"), ("dst", "<u4"), ("orient", "u1"), ("reserved", "u1", (3,)), ("length", "<u8"), ("start", "<u8")])
# ogb_unitig_coverage: the depth of a unitig is bases [start, start + length) of the flat profile (OverlapGraph.depth)
COVERAGE_DTYPE = np.dtype([("edge", "<u4"), ("reads", "<u4"), ("contained", "<u4"), ("depth_min", "<u4"), ("depth_max", "<u4"), ("reserved", "<u4"),
                           ("length", "<u8"), ("start", "<u8"), ("read_count", "<u8"), ("depth_sum", "<u8"), ("depth_sq_sum", "<u8")])
assert CEDGE_DTYPE.itemsize == 40 and CITEM_DTYPE.itemsize == 8 and UNITIG_DTYPE.itemsize == 32 and COVERAGE_DTYPE.itemsize == 64
assert EDGE_DTYPE.itemsize == C.sizeof(Edge) == 12


def _reads_to_buffers(reads):
    """list of str/bytes -> (uint8 bases, uint64 offsets)."""
    bs = [r.encode() if isinstance(r, str) else bytes(r) for r in reads]
    offs = np.zeros(len(bs) + 1, dtype=np.uint64)
    if bs:
        offs[1:] = np.cumsum([len(b) for b in bs], dtype=np.uint64)
    bases = np.frombuffer(b"".join(bs), dtype=np.uint8) if bs else np.zeros(0, dtype=np.uint8)
    return bases, offs


class Dataset:
    """Dataset(pairedEndFileNames, singleEndFileNames, minOverlap) (Dataset.cpp:39-65)."""

    def __init__(self, pairedEndFileNames=(), singleEndFileNames=(), minOverlap=0, reads=None, bases=None, offsets=None, device=None):
        """device: a Context -- canonical strand, sort and dedupe run on that GPU (ogb_dataset_finalize_device) and the
        packed reads stay in its HBM; None: the host threads do it (ogb_dataset_finalize)."""
        self._h = C.c_void_p()
        check(lib().ogb_dataset_create(C.byref(self._h)))
        self.pairedEndDatasetFileNames = list(pairedEndFileNames)
        self.singleEndDatasetFileNames = list(singleEndFileNames)
        for f in self.pairedEndDatasetFileNames + self.singleEndDatasetFileNames:
            check(lib().ogb_dataset_add_file(self._h, str(f).encode()))
        if reads is not None:
            bases, offsets = _reads_to_buffers(reads)
        if bases is not None:
            bases = np.ascontiguousarray(bases, dtype=np.uint8)
            offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
            check(lib().ogb_dataset_add_reads(self._h, bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1))
        if device is not None:
            check(lib().ogb_dataset_finalize_device(self._h, device._h, int(minOverlap)))
        else:
            check(lib().ogb_dataset_finalize(self._h, int(minOverlap)))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().ogb_dataset_destroy(self._h)
            self._h = None

    def getNumberOfReads(self):
        return lib().ogb_dataset_n_reads(self._h)

    def getNumberOfUniqueReads(self):
        return lib().ogb_dataset_n_unique(self._h)

    @property
    def shortestReadLength(self):
        return lib().ogb_dataset_shortest(self._h)

    @property
    def longestReadLength(self):
        return lib().ogb_dataset_longest(self._h)

    @property
    def minimumOverlapLength(self):
        return lib().ogb_dataset_min_overlap(self._h)

    def lengths(self):
        n = self.getNumberOfUniqueReads()
        p = lib().ogb_dataset_lengths(self._h)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint16)), shape=(n,)).copy() if n else np.zeros(0, np.uint16)

    def frequencies(self):
        n = self.getNumberOfUniqueReads()
        p = lib().ogb_dataset_frequencies(self._h)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint32)), shape=(n,)).copy() if n else np.zeros(0, np.uint32)

    def packed(self):
        """(words, word_offsets, lengths) views of the packed store handed to the device."""
        n = self.getNumberOfUniqueReads()
        nw = C.c_uint64()
        pw = lib().ogb_dataset_words(self._h, C.byref(nw))
        po = lib().ogb_dataset_word_offsets(self._h)
        words = np.ctypeslib.as_array(C.cast(pw, C.POINTER(C.c_uint64)), shape=(nw.value,)) if nw.value else np.zeros(0, np.uint64)
        offs = np.ctypeslib.as_array(C.cast(po, C.POINTER(C.c_uint64)), shape=(n + 1,))
        return words, offs, self.lengths()

    def getReadFromID(self, ID, reverse=False):
        """Forward (or reverse-complement) string of read ID (Dataset.cpp:482, Read.h:58-59)."""
        buf = C.create_string_buffer(65536)
        ln = C.c_uint32()
        check(lib().ogb_dataset_get_read(self._h, int(ID), 1 if reverse else 0, buf, 65536, C.byref(ln)))
        return buf.raw[:ln.value].decode()

    def getReadFromString(self, read):
        """ID of a read given its string or reverse complement, 0 if absent (Dataset.cpp:421-455)."""
        out = C.c_uint64()
        b = read.encode() if isinstance(read, str) else bytes(read)
        check(lib().ogb_dataset_find_read(self._h, b, len(b), C.byref(out)))
        return out.value


class Context:
    """One GPU / one rank (ogb_context)."""

    def __init__(self, device=0, rank=0, n_ranks=1, nccl_uid=None):
        self._h = C.c_void_p()
        if n_ranks > 1:
            check(lib().ogb_context_create_dist(C.byref(self._h), device, rank, n_ranks, nccl_uid))
        else:
            check(lib().ogb_context_create(C.byref(self._h), device))

    def close(self):
        if getattr(self, "_h", None):
            lib().ogb_context_destroy(self._h)
            self._h = None

    __del__ = close

    def stats(self):
        s = Stats()
        check(lib().ogb_get_stats(self._h, C.byref(s)))
        return s.as_dict()


def nccl_unique_id():
    buf = C.create_string_buffer(128)
    check(lib().ogb_nccl_unique_id(buf))
    return buf.raw


class HashTable:
    """HashTable() + insertDataset(Dataset*, minOverlapLength) (HashTable.cpp:37-80)."""

    def __init__(self, context=None):
        self.ctx = context if context is not None else Context()
        self.dataSet = None

    def insertDataset(self, d, minOverlapLength):
        self.dataSet = d
        check(lib().ogb_reads_upload_dataset(self.ctx._h, d._h))
        check(lib().ogb_hash_build(self.ctx._h, int(minOverlapLength)))
        return True

    def getHashStringLength(self):
        return lib().ogb_hash_string_length(self.ctx._h)

    def getHashTableSize(self):
        return lib().ogb_hash_table_size(self.ctx._h)

    def getDataset(self):
        return self.dataSet

    def getListOfReads(self, subString):
        """Entries id | orientation<<62 for one key (HashTable.cpp:202-221)."""
        return self.getListsOfReads([subString])[0]

    def getListsOfReads(self, keys):
        h = self.getHashStringLength()
        ks = [k.encode() if isinstance(k, str) else bytes(k) for k in keys]
        assert all(len(k) == h for k in ks), "keys must have hashStringLength bases"
        flat = np.frombuffer(b"".join(ks), dtype=np.uint8) if ks else np.zeros(0, np.uint8)
        offs = np.zeros(len(ks) + 1, dtype=np.uint64)
        cap = max(64, 8 * len(ks))
        while True:
            out = np.zeros(cap, dtype=np.uint64)
            rc = lib().ogb_hash_lookup(self.ctx._h, flat.ctypes.data, len(ks), out.ctypes.data, cap, offs.ctypes.data)
            if rc == 5 and int(offs[-1]) > cap:   # OGB_E_CAPACITY: offsets were still filled in
                cap = int(offs[-1])
                continue
            check(rc)
            break
        return [out[int(offs[i]):int(offs[i + 1])].copy() for i in range(len(ks))]


class OverlapGraph:
    """OverlapGraph(HashTable*) = buildOverlapGraphFromHashTable up to OverlapGraph.cpp:210."""

    def __init__(self, ht, keep_pre=False):
        self.hashTable = ht
        self.ctx = ht.ctx
        self.dataSet = ht.getDataset()
        self.buildOverlapGraphFromHashTable(keep_pre)

    def buildOverlapGraphFromHashTable(self, keep_pre=False):
        self.markContainedReads()
        check(lib().ogb_build_graph(self.ctx._h, 1 if keep_pre else 0))
        return True

    def markContainedReads(self):
        check(lib().ogb_mark_contained(self.ctx._h))

    def superReadIDs(self):
        """Read::superReadID for ids 0..N (entry 0 unused)."""
        n = self.dataSet.getNumberOfUniqueReads()
        out = np.zeros(n + 1, dtype=np.uint64)
        check(lib().ogb_super_read_ids(self.ctx._h, out.ctypes.data, n + 1))
        return out

    def _count(self, which):
        n = C.c_uint64()
        check(lib().ogb_graph_edge_count(self.ctx._h, which, C.byref(n)))
        return n.value

    def getNumberOfEdges(self):
        return self._count(0)

    def getNumberOfNodes(self):
        return self.ctx.stats()["nodes_final"]

    def edges(self, pre=False):
        """Directed edges as a structured array sorted by (src, offset, dst, orient)."""
        which = 1 if pre else 0
        n = self._count(which)
        out = np.zeros(n, dtype=EDGE_DTYPE)
        check(lib().ogb_graph_edges(self.ctx._h, which, out.ctypes.data, n))
        return out

    def edges_shard(self):
        """The post-reduction edges whose source lies in this rank's node range (one rank: all of them)."""
        n = C.c_uint64()
        cap = self._count(0)
        out = np.zeros(cap, dtype=EDGE_DTYPE)
        check(lib().ogb_graph_edges_shard(self.ctx._h, out.ctypes.data, cap, C.byref(n)))
        return out[:n.value]

    def simplify(self):
        """The fix-point that ends buildOverlapGraphFromHashTable (OverlapGraph.cpp:211-215: contractCompositePaths +
        removeDeadEndNodes until neither changes anything), on the device. Returns (edges, items, stats): edges as CEDGE_DTYPE
        records in source order, the reads inside edge i = items[list_start : list_start + count] (CITEM_DTYPE)."""
        from ._lib import SimplifyStats
        st = SimplifyStats()
        check(lib().ogb_graph_simplify(self.ctx._h, C.byref(st)))
        edges = np.zeros(st.n_edges_out, dtype=CEDGE_DTYPE)
        items = np.zeros(st.n_items, dtype=CITEM_DTYPE)
        check(lib().ogb_graph_composite_edges(self.ctx._h, edges.ctypes.data, len(edges), items.ctypes.data, len(items)))
        return edges, items, st.as_dict()

    def spell(self, canonical=True, first=0, count=None):
        """Spells unitigs [first, first + count) of the simplified graph's edges (the canonical ones, src < dst or a self-edge's first
        half, with canonical=True; count None = all) on the device -- the sequences getStringInEdge (OverlapGraph.cpp:2009) returns.
        Needs simplify() first. The result stays on the device; returns the ogb_spell_stats as a dict."""
        from ._lib import SpellStats
        st = SpellStats()
        check(lib().ogb_graph_spell(self.ctx._h, 1 if canonical else 0, int(first), 2**64 - 1 if count is None else int(count), C.byref(st)))
        self._spelled, self._samples = st.as_dict(), 0             # a spell starts a new list of samples (map_reads)
        return st.as_dict()

    def unitigs(self, canonical=True, ascii=True, first=0, count=None):
        """(records, sequences): records as UNITIG_DTYPE in edge order; sequences one flat buffer in which unitig i is
        sequences[start : start + length] -- uint8 ACGT bytes with ascii=True, else the packed uint64 words (2-bit, base p of a
        unitig in bits 63-2(p%32) .. 62-2(p%32) of word start/32 + p/32)."""
        st = self.spell(canonical, first, count)
        recs = np.zeros(st["unitigs"], dtype=UNITIG_DTYPE)
        out = np.zeros(st["words"] * 32, dtype=np.uint8) if ascii else np.zeros(st["words"], dtype=np.uint64)
        check(lib().ogb_graph_unitigs(self.ctx._h, recs.ctypes.data, len(recs), out.ctypes.data, out.nbytes, 1 if ascii else 0))
        return recs, out

    def write_unitigs(self, path, canonical=True):
        """Spells the (canonical) unitigs and writes them as FASTA (ogb_graph_write_unitigs); returns the spell stats."""
        st = self.spell(canonical)
        check(lib().ogb_graph_write_unitigs(self.ctx._h, str(path).encode()))
        return st

    def coverage(self, canonical=True, first=0, count=None):
        """Spells unitigs [first, first + count) (see spell) and computes their per-base read depth on the device, weighted by the
        Dataset's read frequencies, contained reads placed inside their super reads (ogb_graph_coverage). Returns (records as
        COVERAGE_DTYPE in the unitig order, the ogb_coverage_stats as a dict)."""
        from ._lib import CoverageStats
        self.spell(canonical, first, count)
        freq = np.ascontiguousarray(self.dataSet.frequencies(), dtype=np.uint32)
        st = CoverageStats()
        check(lib().ogb_graph_coverage(self.ctx._h, freq.ctypes.data, len(freq), C.byref(st)))
        recs = np.zeros(st.unitigs, dtype=COVERAGE_DTYPE)
        check(lib().ogb_graph_unitig_coverage(self.ctx._h, recs.ctypes.data, len(recs), None, 0))
        return recs, st.as_dict()

    def depth(self, canonical=True, first=0, count=None):
        """(records, depth): as coverage(), plus the uint32 per-base depth in the spell's word-aligned layout -- unitig i is
        depth[start : start + length], the bases up to its next multiple of 32 are 0."""
        recs, _ = self.coverage(canonical, first, count)
        words = int((recs["start"][-1] + recs["length"][-1] + 31) // 32) if len(recs) else 0     # the layout ends with the last unitig
        out = np.zeros(32 * words, dtype=np.uint32)
        check(lib().ogb_graph_unitig_coverage(self.ctx._h, recs.ctypes.data, len(recs), out.ctypes.data, len(out)))
        return recs, out

    def write_coverage(self, path, canonical=True):
        """Computes the coverage of the (canonical) unitigs and writes it as TSV (ogb_graph_write_coverage), one line per unitig
        named as in write_unitigs' FASTA; returns the coverage stats."""
        _, st = self.coverage(canonical)
        check(lib().ogb_graph_write_coverage(self.ctx._h, str(path).encode()))
        return st

    def map_reads(self, reads=None, bases=None, offsets=None, hits=False, max_mismatches=0, strata=False):
        """Maps one sample -- a list of str/bytes reads, or flat ASCII bases + offsets (n + 1) -- onto the unitigs of the last spell()
        (ogb_graph_map_reads_approx): every read that passes the Dataset filter counts 1 on every placement of itself or its reverse
        complement with the fewest substitutions, at most min(max_mismatches, len // K - 1) (K = min(32, minOverlap + 1); 0: exact
        occurrences only). The sample is appended to the samples since that spell. Returns (records as COVERAGE_DTYPE in the unitig
        order: reads = read_count = placements, the ogb_map_stats as a dict[, hits][, strata]): hits = uint32 placements per read,
        OGB_MAP_FILTERED for a filtered read; strata = uint8 substitutions of each read's placements, OGB_MAP_UNPLACED for a read
        that is filtered or not mapped."""
        if reads is not None:
            bases, offsets = _reads_to_buffers(reads)
        if bases is None:
            bases, offsets = np.zeros(0, np.uint8), np.zeros(1, np.uint64)
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        return self._map(bases.ctypes.data, offsets.ctypes.data, len(offsets) - 1, hits, max_mismatches, strata)

    def map_file(self, path, hits=False, max_mismatches=0, strata=False):
        """map_reads() of the reads of a FASTA or FASTQ file, read by the Dataset's parser (ogb_dataset_add_file)."""
        ds = C.c_void_p()
        check(lib().ogb_dataset_create(C.byref(ds)))
        try:
            check(lib().ogb_dataset_add_file(ds, str(path).encode()))
            b, o, n = C.c_void_p(), C.c_void_p(), C.c_uint64()
            check(lib().ogb_dataset_raw_reads(ds, C.byref(b), C.byref(o), C.byref(n)))
            return self._map(b.value, o.value, n.value, hits, max_mismatches, strata)
        finally:
            lib().ogb_dataset_destroy(ds)

    def _map(self, bases, offsets, n, hits, max_mismatches=0, strata=False):
        from ._lib import MapStats
        st = MapStats()
        h = np.zeros(n, np.uint32) if hits else None
        s = np.zeros(n, np.uint8) if strata else None
        check(lib().ogb_graph_map_reads_approx(self.ctx._h, bases, offsets, n, int(max_mismatches), h.ctypes.data if hits else None,
                                               s.ctypes.data if strata else None, C.byref(st)))
        self._samples = st.sample + 1
        recs, _ = self.sample_depth(st.sample, profile=False)
        return (recs, st.as_dict()) + ((h,) if hits else ()) + ((s,) if strata else ())

    def sample_depth(self, sample=-1, profile=True):
        """(records, profile) of a sample mapped since the last spell (-1: the last one): the profile is the uint32 per-base depth in
        the spell's word-aligned layout (unitig i is profile[start : start + length]), kept for the last sample only -- None for
        the others, or with profile=False."""
        n = getattr(self, "_samples", 0)
        j = n + sample if sample < 0 else sample
        recs = np.zeros(self._spelled["unitigs"] if n else 0, dtype=COVERAGE_DTYPE)
        depth = np.zeros(32 * self._spelled["words"], np.uint32) if n and profile and j == n - 1 else None
        check(lib().ogb_graph_sample_coverage(self.ctx._h, max(j, 0), recs.ctypes.data, len(recs), None if depth is None else depth.ctypes.data,
                                              0 if depth is None else len(depth)))
        return recs, depth

    def write_depths(self, path, names=None):
        """Writes the depth table of every sample since the last spell in MetaBAT's layout (ogb_graph_write_depths); names: one per
        sample (None: sample_<j>)."""
        arr = None
        if names is not None:
            if len(names) != getattr(self, "_samples", 0):
                raise ValueError(f"{len(names)} names for {getattr(self, '_samples', 0)} samples")
            arr = (C.c_char_p * len(names))(*[str(x).encode() for x in names])
        check(lib().ogb_graph_write_depths(self.ctx._h, str(path).encode(), arr))

    def checksum(self, pre=False):
        """[xor, sum] of the 64-bit mix of every edge tuple, computed on the device (the figure of tests/golden/full_size.json)."""
        x, t = C.c_uint64(), C.c_uint64()
        check(lib().ogb_graph_checksum(self.ctx._h, 1 if pre else 0, C.byref(x), C.byref(t)))
        return [x.value, t.value]


def edges_as_tuples(e):
    """structured edge array -> (n,4) uint32 [src, dst, offset, orient] (the oracle's tuple layout)."""
    out = np.empty((len(e), 4), dtype=np.uint32)
    out[:, 0], out[:, 1], out[:, 2], out[:, 3] = e["src"], e["dst"], e["offset"], e["orient"]
    return out
