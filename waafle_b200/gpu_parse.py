"""BLAST outfmt-6 text parsed ON THE GPU (csrc/wfl_parse.cu) into the hit columns the packer ships.

Same values as `parsers.read_blast_hits` -- i.e. as the reference's `Hit` objects (waafle/utils.py:192-241) -- but the
per-row work (field split, integer / decimal conversion, scov_modified and waafle_score arithmetic, dictionary coding
of the taxon and of the annotation systems, contig block detection) runs as CUDA kernels over the raw bytes; the host
only touches the DISTINCT names (a few thousand taxa, a handful of systems, one qseqid per contig).  Rows the device
parser cannot reproduce exactly (quoting, exponent floats, malformed rows) make `parse` return None: the caller then
uses the CPU reader, which has the reference's error behaviour.  No CPU fallback is hidden in here.
"""

import ctypes

import numpy as np

from .engine import EngineError, load_library, mark_cuda_touched

TAX_SLOTS, SYS_SLOTS = 1 << 20, 64
_ready = False


def _lib():
    global _ready
    lib = load_library()
    if not _ready:
        P = ctypes.POINTER
        lib.wfl_parser_create.argtypes = [ctypes.c_int, P(ctypes.c_void_p)]
        lib.wfl_parser_destroy.argtypes = [ctypes.c_void_p]
        lib.wfl_parser_destroy.restype = None
        lib.wfl_parser_last_error.argtypes = [ctypes.c_void_p]
        lib.wfl_parser_last_error.restype = ctypes.c_char_p
        lib.wfl_parse_blast.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int64, P(ctypes.c_int32), P(ctypes.c_int64)]
        lib.wfl_parse_blast.restype = ctypes.c_int64
        lib.wfl_parse_blast_resident.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, P(ctypes.c_int32),
                                                 P(ctypes.c_int64)]
        lib.wfl_parse_blast_resident.restype = ctypes.c_int64
        lib.wfl_parser_text.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p]
        lib.wfl_inflate_bgzf.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64,
                                         P(ctypes.c_int64), P(ctypes.c_float), P(ctypes.c_float)]
        lib.wfl_inflate_bgzf.restype = ctypes.c_int64
        lib.wfl_parse_distinct.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_int32]
        lib.wfl_parse_fetch.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 13
        lib.wfl_parser_times.argtypes = [ctypes.c_void_p, P(ctypes.c_float), P(ctypes.c_float), P(ctypes.c_float)]
        lib.wfl_parse_gff.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int64, P(ctypes.c_int32), P(ctypes.c_int64)]
        lib.wfl_parse_gff.restype = ctypes.c_int64
        lib.wfl_parse_gff_fetch.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 7
        lib.wfl_parser_call_genes.argtypes = [ctypes.c_void_p, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                              P(ctypes.c_int64), P(ctypes.c_float)]
        lib.wfl_parser_call_genes.restype = ctypes.c_int64
        lib.wfl_parser_genes_fetch.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 4
        _ready = True
    return lib


class InflateError(EngineError):
    """A BGZF member failed validation on the device (`member`: the first such member of the table)."""

    def __init__(self, member):
        super().__init__("BGZF member {} failed validation on the device".format(member))
        self.member = member


class _TextNames:
    """Subject headers by row, sliced out of the file text on demand (the writer only asks for the winning hits)."""

    def __init__(self, text, off, length):
        self._text, self._off, self._len = text, off, length

    def __len__(self):
        return len(self._off)

    def __getitem__(self, i):
        o = int(self._off[int(i)])
        return self._text[o:o + int(self._len[int(i)])].decode()


class ResidentParse:
    """The device columns a HitTable came from: parse number `generation` of `parser`.  `taxon_slots[k]`: the slot of the
    HitTable's taxon_names[k] in the parser's distinct-taxon set; `sys_perm`: the system map of wfl_parse_fetch (None
    without annotation systems).  packing.pack_resident builds the scoring batch from these columns on the device."""

    def __init__(self, parser, generation, taxon_slots, sys_perm):
        self.parser, self.generation = parser, generation
        self.taxon_slots, self.sys_perm = taxon_slots, sys_perm

    @property
    def live(self):
        """The parser is open and has not parsed anything since."""
        return self.parser.is_open and self.parser.generation == self.generation


def live_resident(hits):
    """The ResidentParse of a HitTable whose parser still holds its columns, else None."""
    r = getattr(hits, "resident", None)
    return r if r is not None and r.live else None


class BlastParser:
    """One parser handle on one GPU.  `generation` counts the parses made with it: the device columns belong to the last
    one only."""

    def __init__(self, device=0):
        self._lib = _lib()
        h = ctypes.c_void_p()
        mark_cuda_touched()
        rc = self._lib.wfl_parser_create(int(device), ctypes.byref(h))
        if rc != 0 or not h:
            raise EngineError("wfl_parser_create(device={}) failed with {}: no usable CUDA device".format(device, rc))
        self._h = h
        self.device = int(device)
        self.generation = 0
        self.times = {}

    @property
    def is_open(self):
        return bool(getattr(self, "_h", None))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.wfl_parser_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc < 0:
            raise EngineError("waafle_b200 parser error {}: {}".format(rc, self._lib.wfl_parser_last_error(self._h).decode()))

    def parse(self, text):
        """`text`: bytes of a whole blastout file (or of whole rows of it).  Returns a parsers.HitTable, or None if some
        row needs the CPU reader."""
        if not isinstance(text, (bytes, bytearray)):
            text = bytes(text)
        flagged, first = ctypes.c_int32(), ctypes.c_int64()
        if len(text.strip()) == 0:   # an empty parse on the device too, so that call_genes sees no blocks
            text = b""
        self.generation += 1
        n = self._lib.wfl_parse_blast(self._h, text, len(text), ctypes.byref(flagged), ctypes.byref(first))
        return self._collect(text, n, flagged)

    def inflate_bgzf(self, comp, members):
        """Inflate BGZF bytes `comp` (member table `members`, compressed.bgzf_members) into the parser's resident text on
        the device.  Returns the text length; raises InflateError when a member fails validation."""
        members = np.ascontiguousarray(members, dtype=np.int64)
        bad, h2d, kern = ctypes.c_int64(), ctypes.c_float(), ctypes.c_float()
        n = self._lib.wfl_inflate_bgzf(self._h, bytes(comp), len(comp), members.ctypes.data_as(ctypes.c_void_p),
                                       len(members), ctypes.byref(bad), ctypes.byref(h2d), ctypes.byref(kern))
        if bad.value >= 0:
            raise InflateError(int(bad.value))
        self._check(n)
        self.inflate_times = dict(ms_h2d=h2d.value, ms_inflate=kern.value, members=len(members), comp_bytes=len(comp),
                                  text_bytes=int(n))
        return int(n)

    def text(self, off, n):
        """Bytes [off, off + n) of the resident text (a bytearray, filled in place)."""
        buf = bytearray(int(n))
        dst = ctypes.addressof((ctypes.c_char * len(buf)).from_buffer(buf)) if len(buf) else None
        self._check(self._lib.wfl_parser_text(self._h, int(off), int(n), dst))
        return buf

    def parse_bgzf(self, comp, members, own=None):
        """Inflate BGZF bytes on the device and parse the text where it lies.  `own` = (offset, length): parse only that
        byte range of the text (whole rows).  Returns the same HitTable as `parse` on the same text, or None if some row
        needs the CPU reader (`text(*own)` then gives the rows); raises InflateError for a member that fails validation."""
        size = self.inflate_bgzf(comp, members)
        off, n = own if own is not None else (0, size)
        text = self.text(off, n)
        if len(text.strip()) == 0:
            off, n = 0, 0
        flagged, first = ctypes.c_int32(), ctypes.c_int64()
        self.generation += 1
        rows = self._lib.wfl_parse_blast_resident(self._h, off, n, ctypes.byref(flagged), ctypes.byref(first))
        hits = self._collect(text if n else b"", rows, flagged)
        if hits is not None:
            self.times.update(self.inflate_times)
        return hits

    def _collect(self, text, n, flagged):
        """The HitTable of the parse that returned `n` rows over host bytes `text` (None: a row needs the CPU reader)."""
        from . import parsers
        self._check(n)
        if flagged.value:
            return None
        if len(text) == 0:
            self.times = dict(ms_h2d=0.0, ms_kernels=0.0, ms_d2h=0.0, rows=0, bytes=0)
            hits = parsers.hits_from_columns(*([[]] * 10))
            hits.resident = ResidentParse(self, self.generation, np.zeros(0, np.int64), None)
            return hits
        n = int(n)
        # ---- the distinct names: taxa (2^20 slots) and annotation systems (64 slots) ----
        vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        th, to, tl = np.empty(TAX_SLOTS, np.uint64), np.empty(TAX_SLOTS, np.int64), np.empty(TAX_SLOTS, np.int32)
        self._check(self._lib.wfl_parse_distinct(self._h, 0, vp(th), vp(to), vp(tl), TAX_SLOTS))
        tslots = np.flatnonzero(th)
        taxon_names = [text[int(o):int(o) + int(l)].decode() for o, l in zip(to[tslots], tl[tslots])]
        if len(set(taxon_names)) != len(taxon_names):
            return None   # two slots, one name: a 64-bit hash collision -- let the CPU reader handle the file
        tlut = np.full(TAX_SLOTS, -1, np.int32)
        tlut[tslots] = np.arange(len(tslots), dtype=np.int32)
        sh, so, sl = np.empty(SYS_SLOTS, np.uint64), np.empty(SYS_SLOTS, np.int64), np.empty(SYS_SLOTS, np.int32)
        self._check(self._lib.wfl_parse_distinct(self._h, 1, vp(sh), vp(so), vp(sl), SYS_SLOTS))
        sslots = np.flatnonzero(sh)
        snames = [text[int(o):int(o) + int(l)].decode() for o, l in zip(so[sslots], sl[sslots])]
        systems = sorted(set(snames))
        if len(systems) != len(snames) or len(systems) > 32:
            return None
        perm = np.full(SYS_SLOTS, -1, np.int32)
        for slot, name in zip(sslots, snames):
            perm[slot] = systems.index(name)
        # ---- the columns ----
        cols = dict(qstart=np.empty(n, np.int32), qend=np.empty(n, np.int32), score=np.empty(n, np.float64),
                    scov=np.empty(n, np.float64), strand=np.empty(n, np.int8), tcode=np.empty(n, np.int32),
                    sysmask=np.empty(n, np.uint32), ss_off=np.empty(n, np.int64), ss_len=np.empty(n, np.int32),
                    newblock=np.empty(n, np.uint8), q_off=np.empty(n, np.int64), q_len=np.empty(n, np.int32))
        self._check(self._lib.wfl_parse_fetch(self._h, vp(perm), *[vp(cols[k]) for k in (
            "qstart", "qend", "score", "scov", "strand", "tcode", "sysmask", "ss_off", "ss_len", "newblock", "q_off", "q_len")]))
        t = [ctypes.c_float() for _ in range(3)]
        self._lib.wfl_parser_times(self._h, *[ctypes.byref(x) for x in t])
        self.times = dict(ms_h2d=t[0].value, ms_kernels=t[1].value, ms_d2h=t[2].value, rows=n, bytes=len(text))
        starts = np.flatnonzero(cols["newblock"]).astype(np.int64)
        block_names = [text[int(o):int(o) + int(l)].decode() for o, l in zip(cols["q_off"][starts], cols["q_len"][starts])]
        names = _TextNames(text, cols["ss_off"], cols["ss_len"])
        hits = parsers.HitTable(
            qseqid=None, qstart=cols["qstart"], qend=cols["qend"], taxon=None, score=cols["score"],
            scov_modified=cols["scov"], strand=cols["strand"], sseqid_id=None, sseqid_names=names,
            sseqid_annotations=parsers._LazyAnnotations(names), systems=systems, sysmask=cols["sysmask"],
            taxon_codes=tlut[cols["tcode"]], taxon_names=taxon_names, block_starts=starts, block_names=block_names)
        hits.resident = ResidentParse(self, self.generation, tslots, perm if systems else None)
        return hits

    def call_genes(self, min_overlap, min_gene_length, min_scov):
        """waafle_genecaller over the hit columns of the last `parse` (still on the device: no hit data is shipped again).
        Returns (gene_off [n_blocks + 1], start, end, strand char codes): the genes of contig block b (the blocks of the
        parse's HitTable.block_starts) are rows gene_off[b] .. gene_off[b + 1]."""
        nb, ms = ctypes.c_int64(), ctypes.c_float()
        n = self._lib.wfl_parser_call_genes(self._h, float(min_overlap), float(min_gene_length), float(min_scov),
                                            ctypes.byref(nb), ctypes.byref(ms))
        self._check(n)
        n = int(n)
        gene_off = np.zeros(nb.value + 1, np.int64)
        start, end, strand = np.empty(n, np.int32), np.empty(n, np.int32), np.empty(n, np.int8)
        vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        self._check(self._lib.wfl_parser_genes_fetch(self._h, vp(gene_off), vp(start), vp(end), vp(strand)))
        self.times["ms_genecall"] = ms.value
        return gene_off, start, end, strand

    def parse_gff(self, text):
        """`text`: bytes of a GFF file.  Returns a parsers.LocusTable (same content as parsers.read_gff_loci), or None if
        some row needs the CPU reader (waafle/utils.py:298-355: 9 fields, integer coordinates, '#' rows skipped)."""
        from . import parsers
        if not isinstance(text, (bytes, bytearray)):
            text = bytes(text)
        if len(text.strip()) == 0:
            return parsers.LocusTable([], [], [], [])
        flagged, first = ctypes.c_int32(), ctypes.c_int64()
        self.generation += 1
        n = self._lib.wfl_parse_gff(self._h, text, len(text), ctypes.byref(flagged), ctypes.byref(first))
        self._check(n)
        if flagged.value:
            return None
        n = int(n)
        vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        cols = dict(start=np.empty(n, np.int32), end=np.empty(n, np.int32), strand=np.empty(n, np.int8),
                    skip=np.empty(n, np.uint8), newblock=np.empty(n, np.uint8), s_off=np.empty(n, np.int64),
                    s_len=np.empty(n, np.int32))
        self._check(self._lib.wfl_parse_gff_fetch(self._h, *[vp(cols[k]) for k in (
            "start", "end", "strand", "skip", "newblock", "s_off", "s_len")]))
        t = [ctypes.c_float() for _ in range(3)]
        self._lib.wfl_parser_times(self._h, *[ctypes.byref(x) for x in t])
        self.times = dict(ms_h2d=t[0].value, ms_kernels=t[1].value, ms_d2h=t[2].value, rows=n, bytes=len(text))
        keep = np.flatnonzero(cols["skip"] == 0)
        nb = cols["newblock"][keep]
        starts = np.flatnonzero(nb)
        names = [text[int(o):int(o) + int(l)].decode() for o, l in zip(cols["s_off"][keep][starts], cols["s_len"][keep][starts])]
        return parsers.LocusTable.from_blocks(names, np.r_[starts, len(keep)], cols["start"][keep], cols["end"][keep],
                                              cols["strand"][keep])
