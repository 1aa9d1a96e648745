"""ctypes binding of the C ABI (include/waafle_b200.h) and the `Engine` host object.

`Engine.score_batch` is the call that replaces the body of the reference's major contig
loop (waafle/waafle_orgscorer.py:952-960).  There is no CPU fallback: if the CUDA library
is missing or no GPU is visible, construction fails loudly.
"""

import ctypes
import os

import numpy as np

from .params import CParams, OrgscorerParams

_LIB_PATH = os.environ.get("WFL_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libwaafle_b200.so")

c_i64p = ctypes.POINTER(ctypes.c_int64)
c_i32p = ctypes.POINTER(ctypes.c_int32)
c_u32p = ctypes.POINTER(ctypes.c_uint32)
c_f64p = ctypes.POINTER(ctypes.c_double)
c_i8p = ctypes.POINTER(ctypes.c_int8)
c_u8p = ctypes.POINTER(ctypes.c_uint8)
c_u16p = ctypes.POINTER(ctypes.c_uint16)

EXPORTS = ["wfl_abi_version", "wfl_device_count", "wfl_create", "wfl_destroy", "wfl_last_error",
           "wfl_set_params", "wfl_set_taxonomy", "wfl_score_batch", "wfl_score_packed", "wfl_upload_batch",
           "wfl_upload_packed", "wfl_run_resident", "wfl_download_results", "wfl_get_stats", "wfl_set_option",
           "wfl_pack_results", "wfl_packed_results_layout", "wfl_debug_gene_scores", "wfl_host_alloc",
           "wfl_host_free", "wfl_parser_create", "wfl_parser_destroy", "wfl_parser_last_error", "wfl_parse_blast",
           "wfl_parse_blast_resident", "wfl_parser_text", "wfl_inflate_bgzf", "wfl_parse_distinct", "wfl_parse_fetch", "wfl_parser_times", "wfl_call_genes", "wfl_download_details", "wfl_parse_gff", "wfl_parse_gff_fetch",
           "wfl_parser_call_genes", "wfl_parser_genes_fetch", "wfl_set_clade_names", "wfl_details_prepare",
           "wfl_details_text", "wfl_debug_format_scores", "wfl_upload_parsed", "wfl_debug_resident_batch"]
ABI_VERSION = 2
_CUDA_TOUCHED = False   # this process has initialised CUDA through the library (a fork could not use it any more)


def mark_cuda_touched():
    global _CUDA_TOUCHED
    _CUDA_TOUCHED = True


def cuda_touched():
    return _CUDA_TOUCHED
PACKED_MAX_NODES, PACKED_MAX_COORD, PACKED_MAX_SYSTEMS = 16384, 65535, 8


class CBatch(ctypes.Structure):
    """`wfl_batch`."""
    _fields_ = [("n_contigs", ctypes.c_int64), ("n_hits", ctypes.c_int64), ("n_loci", ctypes.c_int64),
                ("hit_off", c_i64p), ("locus_off", c_i64p),
                ("hit_qstart", c_i32p), ("hit_qend", c_i32p), ("hit_taxon", c_i32p),
                ("hit_score", c_f64p), ("hit_scov", c_f64p), ("hit_strand", c_i8p),
                ("hit_sysmask", c_u32p),
                ("locus_start", c_i32p), ("locus_end", c_i32p), ("locus_strand", c_i8p)]


class CPackedBatch(ctypes.Structure):
    """`wfl_packed_batch` (compact wire format, 14 B/hit)."""
    _fields_ = [("n_contigs", ctypes.c_int64), ("n_hits", ctypes.c_int64), ("n_loci", ctypes.c_int64),
                ("hit_off", c_i64p), ("locus_off", c_i64p),
                ("hit_qstart16", c_u16p), ("hit_qend16", c_u16p), ("hit_tax16", c_u16p),
                ("hit_score", c_f64p), ("hit_sysmask8", c_u8p),
                ("locus_start", c_i32p), ("locus_end", c_i32p), ("locus_strand", c_i8p)]


class CParsedBatch(ctypes.Structure):
    """`wfl_parsed_batch` (the scoring batch built from a parser's device columns)."""
    _fields_ = [("n_contigs", ctypes.c_int64), ("n_hits", ctypes.c_int64), ("n_loci", ctypes.c_int64),
                ("hit_off", c_i64p), ("hit_src", c_i64p), ("slot_node", c_i32p), ("sys_perm", c_i32p),
                ("locus_off", c_i64p), ("locus_start", c_i32p), ("locus_end", c_i32p), ("locus_strand", c_i8p)]


class CResults(ctypes.Structure):
    """`wfl_results`."""
    _fields_ = [("call", c_u8p), ("direction", c_u8p), ("lifts", c_i32p), ("clade1", c_i32p),
                ("clade2", c_i32p), ("lca", c_i32p), ("best1", c_i32p), ("best2", c_i32p),
                ("crit", c_f64p), ("rank", c_f64p), ("member_off", c_i64p),
                ("n_members_a", c_i32p), ("members", c_i32p),
                ("members_capacity", ctypes.c_int64), ("members_used", ctypes.c_int64),
                ("synteny", c_u8p), ("locus_flags", c_u8p), ("ann_winner", c_i32p),
                ("call_counts", c_i64p), ("call_index", c_i64p)]


class CStats(ctypes.Structure):
    """`wfl_stats`."""
    _fields_ = [(k, ctypes.c_int64) for k in
                ("kernel_launches", "contigs", "hits", "loci", "matched_pairs", "groups", "levels",
                 "pairs_tested", "pairs_scored", "workspace_retries", "smem_contigs", "fallback_contigs",
                 "second_pass_contigs")] + \
               [("fallback_reasons", ctypes.c_int64 * 8)] + \
               [(k, ctypes.c_int64) for k in ("guard_trips", "refined_groups", "host_syncs")] + \
               [("phase_cycles", ctypes.c_int64 * 12)] + \
               [(k, ctypes.c_float) for k in ("ms_h2d", "ms_kernels", "ms_d2h", "ms_score_kernel")]


class EngineError(RuntimeError):
    pass


_lib = None


def load_library(path=None):
    """dlopen the engine; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or _LIB_PATH
    if not os.path.exists(path):
        raise EngineError("CUDA engine library not built: {} (run `python -m waafle_b200.build`)"
                          .format(path))
    lib = ctypes.CDLL(path)
    lib.wfl_abi_version.restype = ctypes.c_int
    lib.wfl_device_count.restype = ctypes.c_int
    lib.wfl_create.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]
    lib.wfl_destroy.argtypes = [ctypes.c_void_p]
    lib.wfl_destroy.restype = None
    lib.wfl_last_error.argtypes = [ctypes.c_void_p]
    lib.wfl_last_error.restype = ctypes.c_char_p
    lib.wfl_set_params.argtypes = [ctypes.c_void_p, ctypes.POINTER(CParams)]
    lib.wfl_set_taxonomy.argtypes = [ctypes.c_void_p, ctypes.c_int32, c_i32p, c_i32p, c_i32p, c_u8p,
                                     ctypes.c_int32, ctypes.c_int32]
    lib.wfl_score_batch.argtypes = [ctypes.c_void_p, ctypes.POINTER(CBatch), ctypes.POINTER(CResults)]
    lib.wfl_score_packed.argtypes = [ctypes.c_void_p, ctypes.POINTER(CPackedBatch), ctypes.POINTER(CResults)]
    lib.wfl_upload_batch.argtypes = [ctypes.c_void_p, ctypes.POINTER(CBatch)]
    lib.wfl_upload_packed.argtypes = [ctypes.c_void_p, ctypes.POINTER(CPackedBatch)]
    lib.wfl_run_resident.argtypes = [ctypes.c_void_p]
    lib.wfl_download_results.argtypes = [ctypes.c_void_p, ctypes.POINTER(CResults)]
    lib.wfl_get_stats.argtypes = [ctypes.c_void_p, ctypes.POINTER(CStats)]
    lib.wfl_set_option.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int64]
    lib.wfl_pack_results.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int64),
                                     ctypes.POINTER(ctypes.c_void_p)]
    lib.wfl_packed_results_layout.argtypes = [ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_int64,
                                              ctypes.POINTER(ctypes.c_int64 * 18)]
    lib.wfl_packed_results_layout.restype = ctypes.c_int64
    lib.wfl_debug_gene_scores.argtypes = [ctypes.c_void_p, ctypes.c_int64, c_i32p, c_i32p, c_f64p,
                                          ctypes.c_int64]
    lib.wfl_debug_gene_scores.restype = ctypes.c_int64
    lib.wfl_set_clade_names.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_char_p, c_i64p]
    lib.wfl_details_prepare.argtypes = [ctypes.c_void_p, ctypes.c_int64, c_i32p, ctypes.c_char_p, c_i64p, c_i64p,
                                        ctypes.POINTER(ctypes.c_float)]
    lib.wfl_details_prepare.restype = ctypes.c_int64
    lib.wfl_details_text.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64,
                                     ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    lib.wfl_details_text.restype = ctypes.c_int64
    lib.wfl_debug_format_scores.argtypes = [ctypes.c_void_p, c_f64p, ctypes.c_int64, ctypes.c_void_p, c_i32p]
    lib.wfl_debug_format_scores.restype = ctypes.c_int64
    lib.wfl_upload_parsed.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(CParsedBatch),
                                      ctypes.POINTER(ctypes.c_float)]
    lib.wfl_debug_resident_batch.argtypes = [ctypes.c_void_p, c_i32p, c_i32p, c_i32p, c_f64p, c_f64p, c_i8p, c_u32p]
    lib.wfl_host_alloc.argtypes = [ctypes.c_size_t, ctypes.POINTER(ctypes.c_void_p)]
    lib.wfl_host_free.argtypes = [ctypes.c_void_p]
    lib.wfl_host_free.restype = None
    if path == _LIB_PATH:
        _lib = lib
    return lib


def _ptr(a, ctype):
    return a.ctypes.data_as(ctypes.POINTER(ctype))


def _name_blob(names):
    """Names as one UTF-8 blob plus offsets [n + 1] (name i = blob[off[i]:off[i + 1]])."""
    enc = [str(nm).encode() for nm in names]
    off = np.zeros(len(enc) + 1, np.int64)
    np.cumsum([len(b) for b in enc], out=off[1:])
    return b"".join(enc), off


def _as(a, dtype):
    a = np.asarray(a)
    if a.dtype != dtype or not a.flags.c_contiguous:
        a = np.ascontiguousarray(a, dtype=dtype)
    return a


class PinnedArena:
    """Page-locked host arrays from wfl_host_alloc (freed when the arena is closed)."""

    def __init__(self, lib=None):
        self._lib = lib or load_library()
        self._ptrs = []

    def empty(self, shape, dtype):
        dtype = np.dtype(dtype)
        n = int(np.prod(shape))
        p = ctypes.c_void_p()
        if self._lib.wfl_host_alloc(max(1, n * dtype.itemsize), ctypes.byref(p)) != 0 or not p:
            raise EngineError("wfl_host_alloc failed")
        self._ptrs.append(p)
        buf = (ctypes.c_uint8 * max(1, n * dtype.itemsize)).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)

    def like(self, a):
        out = self.empty(a.shape, a.dtype)
        out[...] = a
        return out

    def close(self):
        for p in self._ptrs:
            self._lib.wfl_host_free(p)
        self._ptrs = []


class Engine:
    """One handle on one GPU."""

    def __init__(self, device=0, params=None, taxonomy=None):
        self._lib = load_library()
        if self._lib.wfl_abi_version() != ABI_VERSION:
            raise EngineError("ABI version mismatch")
        h = ctypes.c_void_p()
        mark_cuda_touched()
        rc = self._lib.wfl_create(int(device), ctypes.byref(h))
        if rc != 0 or not h:
            raise EngineError("wfl_create(device={}) failed with {}: no usable CUDA device "
                              "(this engine has no CPU fallback)".format(device, rc))
        self._h = h
        self.device = device
        self._keep = {}
        self._pinned = None
        self._res_cache = {}
        self.n_systems = 0
        self._clade_names = None        # names of the taxonomy's nodes, uploaded by the first details_text after set_taxonomy
        self.details_times = {}
        self.resident_times = {}        # ms_kernels of the last upload_parsed
        if params is not None:
            self.set_params(params)
        if taxonomy is not None:
            self.set_taxonomy(taxonomy)

    def use_pinned_results(self, on=True):
        """Keep the result arrays in page-locked memory and reuse them between calls (the arrays a
        call returns are then overwritten by the next call)."""
        if on and self._pinned is None:
            self._pinned = PinnedArena(self._lib)
        if not on and self._pinned is not None:
            self._pinned.close()
            self._pinned = None
        self._res_cache = {}

    def close(self):
        if getattr(self, "_pinned", None):
            self._pinned.close()
            self._pinned = None
        if getattr(self, "_h", None):
            self._lib.wfl_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise EngineError("waafle_b200 engine error {}: {}".format(
                rc, self._lib.wfl_last_error(self._h).decode()))

    # ------------------------------------------------------------------
    def set_option(self, name, value):
        """Tuning / test knobs by name (include/waafle_b200.h: wfl_set_option), e.g. exact=1."""
        self._check(self._lib.wfl_set_option(self._h, name.encode(), int(value)))

    def set_params(self, params):
        if isinstance(params, dict):
            params = OrgscorerParams(**params)
        self.n_systems = params.n_systems
        cp = params.as_ctypes()
        self._check(self._lib.wfl_set_params(self._h, ctypes.byref(cp)))

    def set_taxonomy(self, tax):
        """`tax`: taxonomy.Taxonomy (built) or the dict of its tables()."""
        t = tax.tables() if hasattr(tax, "tables") else tax
        parent, depth = _as(t["parent"], np.int32), _as(t["depth"], np.int32)
        leaf, listed = _as(t["leaf_count"], np.int32), _as(t["listed"], np.uint8)
        self._check(self._lib.wfl_set_taxonomy(
            self._h, len(parent), _ptr(parent, ctypes.c_int32), _ptr(depth, ctypes.c_int32),
            _ptr(leaf, ctypes.c_int32), _ptr(listed, ctypes.c_uint8),
            int(t["root_idx"]), int(t["unknown_idx"])))
        self._clade_names = (list(tax.names), False) if getattr(tax, "names", None) is not None else None

    # ------------------------------------------------------------------
    def _cbatch(self, batch):
        """ctypes view of a batch in either wire format; returns (struct, n, nh, nl, packed)."""
        a = batch.arrays() if hasattr(batch, "arrays") else batch
        packed = "hit_tax16" in a
        if packed:
            spec = dict(hit_off=np.int64, locus_off=np.int64, hit_qstart16=np.uint16, hit_qend16=np.uint16,
                        hit_tax16=np.uint16, hit_score=np.float64, locus_start=np.int32, locus_end=np.int32,
                        locus_strand=np.int8)
            mask_name, mask_dtype, cls = "hit_sysmask8", np.uint8, CPackedBatch
        else:
            spec = dict(hit_off=np.int64, locus_off=np.int64, hit_qstart=np.int32, hit_qend=np.int32,
                        hit_taxon=np.int32, hit_score=np.float64, hit_scov=np.float64, hit_strand=np.int8,
                        locus_start=np.int32, locus_end=np.int32, locus_strand=np.int8)
            mask_name, mask_dtype, cls = "hit_sysmask", np.uint32, CBatch
        k = {name: _as(a[name], dt) for name, dt in spec.items()}
        n, nh, nl = len(k["hit_off"]) - 1, len(k["hit_score"]), len(k["locus_start"])
        cb = cls(n_contigs=n, n_hits=nh, n_loci=nl)
        ftypes = dict(cls._fields_)
        for name, arr in k.items():
            setattr(cb, name, _ptr(arr, ftypes[name]._type_))
        if self.n_systems > 0:
            if a.get(mask_name) is None:
                raise EngineError("params.n_systems > 0 but the batch has no " + mask_name)
            k[mask_name] = _as(a[mask_name], mask_dtype)
            setattr(cb, mask_name, _ptr(k[mask_name], ftypes[mask_name]._type_))
        self._keep = k   # keep the arrays alive while the C side reads them
        return cb, n, nh, nl, packed

    def _alloc_results(self, n, nl, members_capacity):
        S = self.n_systems
        if self._pinned is not None:
            key = (n, nl, S, max(1, members_capacity))
            if key not in self._res_cache:
                # a new shape: the previous shape's page-locked buffers go back first (arrays handed out by earlier calls
                # are documented to die with the next call), so a long-lived engine does not accumulate pinned memory
                self._res_cache = {}
                self._pinned.close()
                e = self._pinned.empty
                self._res_cache = {key: dict(
                    call=e(n, np.uint8), direction=e(n, np.uint8), lifts=e(n, np.int32), clade1=e(n, np.int32),
                    clade2=e(n, np.int32), lca=e(n, np.int32), best1=e(n, np.int32), best2=e(n, np.int32),
                    crit=e(n, np.float64), rank=e(n, np.float64), member_off=e(n + 1, np.int64),
                    n_members_a=e(n, np.int32), members=e(max(1, members_capacity), np.int32),
                    synteny=e(nl, np.uint8), locus_flags=e(nl, np.uint8), ann_winner=e((nl, S), np.int32),
                    call_counts=e(3, np.int64), call_index=e(n, np.int64))}
            r = dict(self._res_cache[key])
            cr = CResults(members_capacity=len(r["members"]), members_used=0)
            for name, arr in r.items():
                setattr(cr, name, _ptr(arr, dict(CResults._fields_)[name]._type_))
            return r, cr
        r = dict(
            call=np.empty(n, np.uint8), direction=np.empty(n, np.uint8),
            lifts=np.empty(n, np.int32), clade1=np.empty(n, np.int32),
            clade2=np.empty(n, np.int32), lca=np.empty(n, np.int32), best1=np.empty(n, np.int32),
            best2=np.empty(n, np.int32), crit=np.empty(n, np.float64), rank=np.empty(n, np.float64),
            member_off=np.empty(n + 1, np.int64), n_members_a=np.empty(n, np.int32),
            members=np.empty(max(1, members_capacity), np.int32),
            synteny=np.empty(nl, np.uint8), locus_flags=np.empty(nl, np.uint8),
            ann_winner=np.empty((nl, S), np.int32),
            call_counts=np.empty(3, np.int64), call_index=np.empty(n, np.int64))
        cr = CResults(members_capacity=len(r["members"]), members_used=0)
        for name, arr in r.items():
            setattr(cr, name, _ptr(arr, dict(CResults._fields_)[name]._type_))
        return r, cr

    def _finish(self, r, cr):
        r["members"] = r["members"][:cr.members_used]
        return r

    def score_batch(self, batch):
        """Host arrays in, host arrays out (H2D + kernels + D2H inside the call).  A packing.ResidentBatch has its hit
        columns built on the device from its parser's columns instead (upload_parsed, run_resident, download)."""
        if hasattr(batch, "hit_src"):
            self.upload_parsed(batch)
            self.run_resident()
            return self.download()
        cb, n, nh, nl, packed = self._cbatch(batch)
        call = self._lib.wfl_score_packed if packed else self._lib.wfl_score_batch
        cap = max(4 * n, 1024)
        for _ in range(2):
            r, cr = self._alloc_results(n, nl, cap)
            rc = call(self._h, ctypes.byref(cb), ctypes.byref(cr))
            if rc == -4:   # WFL_ERR_CAPACITY: results are resident, fetch with a larger buffer
                cap = int(cr.members_used)
                r, cr = self._alloc_results(n, nl, cap)
                rc = self._lib.wfl_download_results(self._h, ctypes.byref(cr))
            self._check(rc)
            return self._finish(r, cr)

    def upload(self, batch):
        cb, n, nh, nl, packed = self._cbatch(batch)
        call = self._lib.wfl_upload_packed if packed else self._lib.wfl_upload_batch
        self._check(call(self._h, ctypes.byref(cb)))
        self._resident = (n, nl)

    def upload_parsed(self, batch):
        """Build the resident wide batch of a packing.ResidentBatch on the device (wfl_upload_parsed) from the columns
        its GPU parse left there; raises EngineError when that parse is no longer live (the parser was closed or has
        parsed again since)."""
        res = batch.resident
        if res is None or not res.live:
            raise EngineError("the batch's GPU parse is no longer live (its parser was closed or parsed again)")
        k = dict(hit_off=_as(batch.hit_off, np.int64), hit_src=_as(batch.hit_src, np.int64),
                 slot_node=_as(batch.slot_node, np.int32), locus_off=_as(batch.locus_off, np.int64),
                 locus_start=_as(batch.locus_start, np.int32), locus_end=_as(batch.locus_end, np.int32),
                 locus_strand=_as(batch.locus_strand, np.int8))
        n, nl = len(k["hit_off"]) - 1, len(k["locus_start"])
        pb = CParsedBatch(n_contigs=n, n_hits=int(k["hit_off"][-1]), n_loci=nl)
        ftypes = dict(CParsedBatch._fields_)
        for name, arr in k.items():
            setattr(pb, name, _ptr(arr, ftypes[name]._type_))
        if res.sys_perm is not None:
            k["sys_perm"] = _as(res.sys_perm, np.int32)
            pb.sys_perm = _ptr(k["sys_perm"], ctypes.c_int32)
        self._keep = k
        ms = ctypes.c_float()
        self._check(self._lib.wfl_upload_parsed(self._h, res.parser._h, ctypes.byref(pb), ctypes.byref(ms)))
        self.resident_times = dict(ms_kernels=ms.value)
        self._resident = (n, nl)

    def debug_resident_batch(self):
        """The hit columns of the resident wide batch (test hook), as Batch.arrays() names them."""
        nh = int(self._keep["hit_off"][-1]) if "hit_off" in self._keep else 0
        out = dict(hit_qstart=np.empty(nh, np.int32), hit_qend=np.empty(nh, np.int32), hit_taxon=np.empty(nh, np.int32),
                   hit_score=np.empty(nh, np.float64), hit_scov=np.empty(nh, np.float64), hit_strand=np.empty(nh, np.int8))
        if self.n_systems > 0:
            out["hit_sysmask"] = np.empty(nh, np.uint32)
        self._check(self._lib.wfl_debug_resident_batch(
            self._h, *[_ptr(out[k], t) for k, t in (("hit_qstart", ctypes.c_int32), ("hit_qend", ctypes.c_int32),
                                                    ("hit_taxon", ctypes.c_int32), ("hit_score", ctypes.c_double),
                                                    ("hit_scov", ctypes.c_double), ("hit_strand", ctypes.c_int8))],
            _ptr(out["hit_sysmask"], ctypes.c_uint32) if "hit_sysmask" in out else None))
        return out

    def run_resident(self):
        self._check(self._lib.wfl_run_resident(self._h))

    def download(self):
        n, nl = self._resident
        r, cr = self._alloc_results(n, nl, max(4 * n, 1024))
        rc = self._lib.wfl_download_results(self._h, ctypes.byref(cr))
        if rc == -4:
            r, cr = self._alloc_results(n, nl, int(cr.members_used))
            rc = self._lib.wfl_download_results(self._h, ctypes.byref(cr))
        self._check(rc)
        return self._finish(r, cr)

    def score_batch_device(self, batch):
        """Plugin call that leaves the results on the device (multi-GPU: they are gathered with NCCL from there)."""
        cb, n, nh, nl, packed = self._cbatch(batch)
        call = self._lib.wfl_score_packed if packed else self._lib.wfl_score_batch
        self._check(call(self._h, ctypes.byref(cb), None))
        self._resident = (n, nl)

    def pack_results(self):
        """The compacted results of the last run as ONE device buffer: (device pointer, bytes, cudaStream_t)."""
        p, nb, st = ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_void_p()
        self._check(self._lib.wfl_pack_results(self._h, ctypes.byref(p), ctypes.byref(nb), ctypes.byref(st)))
        return p.value, nb.value, st.value

    def score_batch_details(self, batch, download=True):
        """--write-details: (results, details) where details = dict of arrays contig / iteration / clade / locus / score --
        every gene score of every clade at every evaluated level (exact pipeline; see include/waafle_b200.h).  With
        download=False the dump stays on the device (details_text reads it there), details is None and the engine keeps
        recording details until set_option("details", 0)."""
        self.set_option("details", 0)
        self.set_option("exact", 1)
        self.score_batch(batch)
        st = self.stats()
        cap = int(st["groups"]) + int(st["levels"]) * 64 + 4096
        lib = self._lib
        P = ctypes.POINTER
        lib.wfl_download_details.restype = ctypes.c_int64
        lib.wfl_download_details.argtypes = [ctypes.c_void_p, P(ctypes.c_int32), P(ctypes.c_int32), P(ctypes.c_int32),
                                             P(ctypes.c_int32), P(ctypes.c_double), ctypes.c_int64]
        for _ in range(4):
            self.set_option("details", cap)
            res = self.score_batch(batch)
            if not download:
                n = lib.wfl_download_details(self._h, None, None, None, None, None, 0)
                self._check(min(int(n), 0))
                if n <= cap:
                    return res, None
                cap = int(n) + 4096
                continue
            d = dict(contig=np.empty(cap, np.int32), iteration=np.empty(cap, np.int32), clade=np.empty(cap, np.int32),
                     locus=np.empty(cap, np.int32), score=np.empty(cap, np.float64))
            n = lib.wfl_download_details(self._h, _ptr(d["contig"], ctypes.c_int32), _ptr(d["iteration"], ctypes.c_int32),
                                         _ptr(d["clade"], ctypes.c_int32), _ptr(d["locus"], ctypes.c_int32),
                                         _ptr(d["score"], ctypes.c_double), cap)
            self._check(min(int(n), 0))
            if n <= cap:
                self.set_option("details", 0)
                return res, {k: v[:int(n)] for k, v in d.items()}
            cap = int(n) + 4096
        raise EngineError("details dump keeps overflowing")

    def details_text(self, order, contig_names, piece_bytes=256 << 20):
        """The --write-details rows of the last score_batch_details run, built on the device, as bytes pieces of at most
        `piece_bytes` each (a contig's rows are never split, so a contig larger than that is one piece).  `order`: contig
        indices of the batch in output order; `contig_names`: the batch's contig names by index.  Needs a taxonomy with
        names (taxonomy.Taxonomy).  Times of the last call land in `details_times` (ms)."""
        if self._clade_names is None:
            raise EngineError("details_text needs the node names of the taxonomy (set_taxonomy with a Taxonomy)")
        names, sent = self._clade_names
        if not sent:
            blob, off = _name_blob(names)
            self._check(self._lib.wfl_set_clade_names(self._h, len(names), blob, _ptr(off, ctypes.c_int64)))
            self._clade_names = (names, True)
        order = _as(order, np.int32)
        blob, off = _name_blob(contig_names)
        before = np.zeros(len(order) + 1, np.int64)
        ms = ctypes.c_float()
        total = self._lib.wfl_details_prepare(self._h, len(order), _ptr(order, ctypes.c_int32), blob,
                                              _ptr(off, ctypes.c_int64), _ptr(before, ctypes.c_int64), ctypes.byref(ms))
        self._check(min(int(total), 0))
        times = dict(ms_length=ms.value, ms_text=0.0, ms_d2h=0.0, bytes=int(total), pieces=0)
        self.details_times = times
        r0, n = 0, len(order)
        buf = None
        while r0 < n:
            # the longest run of contigs from r0 whose rows fit one piece (at least one contig)
            r1 = max(r0 + 1, int(np.searchsorted(before, before[r0] + piece_bytes, side="right")) - 1)
            size = int(before[r1] - before[r0])
            if size:
                if buf is None or len(buf) < size:
                    buf = np.empty(max(size, min(int(total), int(piece_bytes))), np.uint8)
                mk, md = ctypes.c_float(), ctypes.c_float()
                got = self._lib.wfl_details_text(self._h, r0, r1, buf.ctypes.data, len(buf), ctypes.byref(mk), ctypes.byref(md))
                self._check(min(int(got), 0))
                if got != size:
                    raise EngineError("details text: {} bytes, expected {}".format(got, size))
                times["ms_text"] += mk.value
                times["ms_d2h"] += md.value
                times["pieces"] += 1
                yield buf[:size].tobytes()
            r0 = r1

    def debug_format_scores(self, x):
        """The details table's "{:.3f}" of every value of `x` (test hook); raises EngineError outside |x| < 2^53."""
        x = _as(x, np.float64)
        text = np.zeros(24 * max(1, len(x)), np.uint8)
        lens = np.zeros(max(1, len(x)), np.int32)
        self._check(min(int(self._lib.wfl_debug_format_scores(self._h, _ptr(x, ctypes.c_double), len(x), text.ctypes.data,
                                                                _ptr(lens, ctypes.c_int32))), 0))
        raw = text.tobytes()
        return [raw[24 * i:24 * i + int(lens[i])].decode() for i in range(len(x))]

    def stats(self):
        s = CStats()
        self._check(self._lib.wfl_get_stats(self._h, ctypes.byref(s)))
        d = {k: getattr(s, k) for k, _ in CStats._fields_}
        d["phase_cycles"] = list(d["phase_cycles"])
        d["fallback_reasons"] = list(d["fallback_reasons"])
        return d

    def debug_gene_scores(self, contig, capacity=1 << 16):
        """Level-0 gene scores of one contig of the resident batch: (clade, locus, score)."""
        cl, lo, sc = (np.empty(capacity, np.int32), np.empty(capacity, np.int32),
                      np.empty(capacity, np.float64))
        m = self._lib.wfl_debug_gene_scores(self._h, int(contig), _ptr(cl, ctypes.c_int32),
                                            _ptr(lo, ctypes.c_int32), _ptr(sc, ctypes.c_double),
                                            capacity)
        if m < 0:
            self._check(int(m))
        if m > capacity:
            return self.debug_gene_scores(contig, int(m))
        return cl[:m], lo[:m], sc[:m]


_SECTIONS = [("call", np.uint8), ("direction", np.uint8), ("lifts", np.int32), ("clade1", np.int32),
             ("clade2", np.int32), ("lca", np.int32), ("best1", np.int32), ("best2", np.int32),
             ("crit", np.float64), ("rank", np.float64), ("member_off", np.int64), ("n_members_a", np.int32),
             ("members", np.int32), ("synteny", np.uint8), ("locus_flags", np.uint8), ("ann_winner", np.int32),
             ("call_counts", np.int64), ("call_index", np.int64)]


def results_layout(n, nl, S, members):
    """Byte offsets of the 18 sections of a packed results buffer and its total size (wfl_packed_results_layout)."""
    off = (ctypes.c_int64 * 18)()
    total = load_library().wfl_packed_results_layout(n, nl, S, members, ctypes.byref(off))
    return list(off), int(total)


def unpack_results(blob):
    """Host copy of a packed results buffer (uint8 array) -> the dict Engine.score_batch returns."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    n, nl, S, members = (int(x) for x in blob[:32].view(np.int64))
    off, total = results_layout(n, nl, S, members)
    counts = dict(call=n, direction=n, lifts=n, clade1=n, clade2=n, lca=n, best1=n, best2=n, crit=n, rank=n,
                  member_off=n + 1, n_members_a=n, members=members, synteny=nl, locus_flags=nl,
                  ann_winner=nl * S, call_counts=3, call_index=n)
    out = {}
    for (name, dt), o in zip(_SECTIONS, off):
        cnt = counts[name]
        out[name] = blob[o:o + cnt * np.dtype(dt).itemsize].view(dt).copy()
    out["ann_winner"] = out["ann_winner"].reshape(nl, S)
    return out
