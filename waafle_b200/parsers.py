"""BLAST outfmt-6 and GFF readers producing column arrays (the values the packer ships).

Same field lists, derived quantities and error behaviour as the reference's row
objects -- `Hit` (waafle/utils.py:192-241) and `Locus` (waafle/utils.py:298-322) --
but columnar: one numpy array per attribute instead of one Python object per row.
The arithmetic keeps the reference's operation order so that `scov_modified` and
`waafle_score` are bit-identical (UT:216-229).
"""

import csv
import io

import numpy as np
import pandas as pd

try:   # Arrow's CSV reader and string kernels (multi-threaded, no per-row Python objects); optional
    import pyarrow as pa
    import pyarrow.compute as pc
    import pyarrow.csv as pacsv
except Exception:   # pragma: no cover
    pa = pc = pacsv = None

from .utils import die, say, try_open

# UT:167-183
BLAST_FIELDS = ["qseqid", "sseqid", "qlen", "slen", "length", "qstart", "qend", "sstart",
                "send", "pident", "positive", "gaps", "evalue", "bitscore", "sstrand"]
_BLAST_STR = {"qseqid", "sseqid", "sstrand"}
_BLAST_FLOAT = {"pident", "evalue", "bitscore"}
# UT:282-292
GFF_FIELDS = ["seqname", "source", "feature", "start", "end", "score", "strand", "frame",
              "attribute"]

STRAND_PLUS, STRAND_MINUS = ord("+"), ord("-")


class HitTable:
    """All hits of a blastout file, in file order."""

    def __init__(self, qseqid, qstart, qend, taxon, score, scov_modified, strand,
                 sseqid_id, sseqid_names, sseqid_annotations, systems, sysmask,
                 taxon_codes=None, taxon_names=None, qseqid_codes=None, qseqid_names=None,
                 block_starts=None, block_names=None):
        self._qseqid = qseqid               # object array of contig names (None: see block_starts)
        self.qstart = qstart                # int32
        self.qend = qend                    # int32
        self._taxon = taxon                 # object array of taxon names (sseqid field 1; None: see taxon_codes)
        self.score = score                  # float64  waafle_score      UT:229
        self.scov_modified = scov_modified  # float64                    UT:227
        self.strand = strand                # int8 '+' / '-'             UT:214
        self.sseqid_id = sseqid_id          # int32 index into the unique-sseqid tables
        self.sseqid_names = sseqid_names
        self.sseqid_annotations = sseqid_annotations   # list of {system: value}  UT:237-241
        self.systems = systems              # sorted annotation systems seen in the hits
        self.sysmask = sysmask              # uint32 bit s = hit carries systems[s]
        # dictionary-encoded views of `taxon` / `qseqid` (None when built without Arrow): the packer maps the
        # few distinct names once instead of looking every row up
        self.taxon_codes, self.taxon_names = taxon_codes, taxon_names
        self.qseqid_codes, self.qseqid_names = qseqid_codes, qseqid_names
        # run-length view of `qseqid` (GPU parser): rows block_starts[b] .. block_starts[b+1] share block_names[b]
        self.block_starts, self.block_names = block_starts, block_names
        # the GPU parse whose device columns hold these hits (gpu_parse.ResidentParse), or None
        self.resident = None

    def __len__(self):
        return len(self.qstart)

    @property
    def qseqid(self):
        if self._qseqid is None and self.block_starts is not None:
            lens = np.diff(np.r_[self.block_starts, len(self)])
            self._qseqid = np.repeat(np.array(self.block_names, dtype=object), lens)
        return self._qseqid

    @property
    def taxon(self):
        if self._taxon is None and self.taxon_codes is not None:
            self._taxon = (np.array(self.taxon_names, dtype=object)[self.taxon_codes] if len(self.taxon_codes)
                           else np.array([], dtype=object))
        return self._taxon

    def distinct_taxa(self):
        """The taxon names seen in the hits (what Taxonomy.build needs), without a per-row object array."""
        return set(self.taxon_names) if self.taxon_names is not None else set(self.taxon)


def hits_from_columns(qseqid, sseqid, qlen, slen, qstart, qend, sstart, send, pident, sstrand):
    """Derive the engine-facing hit columns from raw BLAST columns (UT:207-241)."""
    qlen, slen, qstart, qend, sstart, send = (
        np.asarray(a, dtype=np.int64) for a in (qlen, slen, qstart, qend, sstart, send))
    pident = np.asarray(pident, dtype=np.float64)
    is_arrow = lambda x: pa is not None and isinstance(x, (pa.Array, pa.ChunkedArray))
    if is_arrow(sstrand):
        minus = pc.equal(sstrand, "minus").to_numpy(zero_copy_only=False).astype(bool)   # UT:214
    else:
        minus = np.asarray(sstrand) == "minus"                   # UT:214
    s1 = np.where(minus, slen - sstart + 1, sstart)              # UT:219-224
    s2 = np.where(minus, slen - send + 1, send)
    ltrim = np.maximum(0, s1 - qstart)                           # UT:225
    rtrim = np.maximum(0, slen - s1 - qlen + qstart)             # UT:226
    denom = slen - ltrim - rtrim
    if np.any(denom == 0):
        raise ZeroDivisionError("float division by zero")       # what UT:227 raises
    scov_modified = (s2 - s1 + 1) / denom.astype(np.float64)     # UT:227
    score = scov_modified * pident / 100.0                       # UT:229
    # subject header: geneid|taxon|system=value...   UT:231-241
    n_rows = len(qstart)
    if is_arrow(sseqid):
        parsed = _parse_subject_headers_arrow(sseqid)
        if parsed is None:
            parsed = _parse_subject_headers_python(np.array(sseqid.to_pylist(), dtype=object))
    else:
        sseqid = np.asarray(sseqid, dtype=object)
        parsed = _parse_subject_headers_arrow(sseqid) if pa is not None and n_rows else None
        if parsed is None:
            parsed = _parse_subject_headers_python(sseqid)
    uniq, inv, taxa, anns, systems, umask, tcodes, tnames = parsed
    qcodes = qnames = None
    if pa is not None and n_rows:
        try:
            qarr = qseqid if is_arrow(qseqid) else pa.array(np.asarray(qseqid, dtype=object), type=pa.string())
            if isinstance(qarr, pa.ChunkedArray):
                qarr = qarr.combine_chunks()
            qenc = qarr.dictionary_encode()
            qcodes = qenc.indices.to_numpy(zero_copy_only=False).astype(np.int32)
            qnames = qenc.dictionary.to_pylist()
        except Exception:
            qcodes = qnames = None
    if is_arrow(qseqid):   # row names as an object array that shares one str per distinct contig
        qseqid = (np.array(qnames, dtype=object)[qcodes] if qcodes is not None
                  else np.array(qseqid.to_pylist(), dtype=object))
    lim = np.iinfo(np.int32)
    if len(qstart) and (max(qstart.max(), qend.max()) > lim.max or min(qstart.min(), qend.min()) < lim.min):
        die("hit coordinates exceed 32 bits")
    return HitTable(
        qseqid=np.asarray(qseqid, dtype=object),
        qstart=qstart.astype(np.int32), qend=qend.astype(np.int32),
        taxon=taxa[inv] if len(inv) else np.array([], dtype=object),
        score=score, scov_modified=scov_modified,
        strand=np.where(minus, STRAND_MINUS, STRAND_PLUS).astype(np.int8),
        sseqid_id=inv.astype(np.int32), sseqid_names=uniq, sseqid_annotations=anns,
        systems=systems,
        sysmask=(umask[inv] if len(inv) else np.array([], dtype=np.uint64)).astype(np.uint32)
        if len(systems) <= 32 else None,
        taxon_codes=tcodes, taxon_names=tnames, qseqid_codes=qcodes, qseqid_names=qnames,
    )


def _parse_annotations(name):
    """{system: value} of one subject header (UT:237-241)."""
    d = {}
    for k in name.split("|")[2:]:
        system, value = k.split("=")
        d[system] = value
    return d


class _ArrowNames:
    """Read-only sequence view of an Arrow string array (no per-row Python objects until asked for)."""

    def __init__(self, arr):
        self._arr = arr

    def __len__(self):
        return len(self._arr)

    def __getitem__(self, i):
        return self._arr[int(i)].as_py()

    def __iter__(self):
        return (x.as_py() for x in self._arr)


class _LazyAnnotations:
    """sseqid_annotations[i] parsed on demand: the writer only asks for the winning hits."""

    def __init__(self, names):
        self._names = names

    def __len__(self):
        return len(self._names)

    def __getitem__(self, i):
        return _parse_annotations(self._names[i])


def _parse_subject_headers_python(sseqid):
    """The row-object way (one split per distinct header); reference error behaviour."""
    if len(sseqid):
        uniq, inv = np.unique(sseqid.astype(str), return_inverse=True)
    else:
        uniq, inv = np.array([], dtype=str), np.array([], dtype=np.int64)
    taxa, anns = [], []
    for name in uniq:
        items = name.split("|")
        if len(items) < 2:
            die("bad subject id header:", name)
        taxa.append(items[1])
        anns.append(_parse_annotations(name))
    systems = sorted({s for d in anns for s in d})
    sysbit = {s: i for i, s in enumerate(systems)}
    umask = np.array([sum(1 << sysbit[s] for s in d) for d in anns] or [0], dtype=np.uint64)
    return list(uniq), inv, np.array(taxa, dtype=object), anns, systems, umask, None, None


def _parse_subject_headers_arrow(sseqid):
    """Same result with Arrow string kernels over the DISTINCT headers; None = let the Python path decide
    (irregular annotation items, for which the reference raises)."""
    try:
        arr = sseqid if isinstance(sseqid, (pa.Array, pa.ChunkedArray)) else pa.array(sseqid, type=pa.string())
        if isinstance(arr, pa.ChunkedArray):
            arr = arr.combine_chunks()
        enc = arr.dictionary_encode()
    except Exception:
        return None
    uniq = enc.dictionary
    inv = enc.indices.to_numpy(zero_copy_only=False).astype(np.int64)
    parts = pc.split_pattern(uniq, "|")
    nparts = pc.list_value_length(parts).to_numpy(zero_copy_only=False).astype(np.int64)
    if len(nparts) and nparts.min() < 2:
        die("bad subject id header:", uniq[int(np.argmax(nparts < 2))].as_py())
    off = parts.offsets.to_numpy(zero_copy_only=False).astype(np.int64)
    flat = parts.values
    tenc = flat.take(pa.array(off[:-1] + 1)).dictionary_encode()
    tnames = tenc.dictionary.to_pylist()
    tcodes_u = tenc.indices.to_numpy(zero_copy_only=False).astype(np.int32)
    # annotation items: list elements 2.. of every distinct header
    n_items = nparts - 2
    total = int(n_items.sum())
    umask = np.zeros(max(len(uniq), 1), dtype=np.uint64)
    systems = []
    if total:
        first = np.repeat(off[:-1] + 2, n_items)
        within = np.arange(total, dtype=np.int64) - np.repeat(np.cumsum(n_items) - n_items, n_items)
        items = flat.take(pa.array(first + within))
        n_eq = pc.count_substring(items, "=")
        if pc.min(n_eq).as_py() != 1 or pc.max(n_eq).as_py() != 1:
            return None
        senc = pc.list_element(pc.split_pattern(items, "="), 0).dictionary_encode()
        snames = senc.dictionary.to_pylist()
        scodes = senc.indices.to_numpy(zero_copy_only=False).astype(np.int64)
        systems = sorted(snames)
        rank = np.array([systems.index(x) for x in snames], dtype=np.uint64)
        if len(systems) <= 64:
            # items are grouped by header: OR the system bits of each header's stretch
            has = np.nonzero(n_items > 0)[0]
            seg = (np.cumsum(n_items) - n_items)[has]
            umask[has] = np.bitwise_or.reduceat(np.uint64(1) << rank[scodes], seg)
    names = _ArrowNames(uniq)
    taxa_u = np.array(tnames, dtype=object)[tcodes_u] if len(tcodes_u) else np.array([], dtype=object)
    return (names, inv, taxa_u, _LazyAnnotations(names), systems, umask,
            tcodes_u[inv] if len(inv) else None, tnames)


def read_blast_hits(path, device=None):
    """Parse a waafle_search blastout file (15-field outfmt 6, UT:167-186).  With `device` (a CUDA device index) the rows
    are parsed on the GPU (gpu_parse.BlastParser); files it cannot reproduce exactly fall through to the CPU reader."""
    if device is not None:
        hits = _gpu_parse_blast(path, device)
        if hits is not None:
            return hits
    want = ("qseqid", "sseqid", "qlen", "slen", "qstart", "qend", "sstart", "send", "pident", "sstrand")
    cols, ok, text = None, False, None
    if pacsv is not None:
        # Arrow: multi-threaded tokeniser (inflates .gz / .bz2 by extension), correctly rounded float conversion
        # (the same doubles as float()); strings stay Arrow arrays -- no per-row Python objects
        try:
            with try_open(path) as fh:   # same "Can't open file" behaviour as the reference
                pass
            types = {f: (pa.string() if f in _BLAST_STR else pa.float64() if f in _BLAST_FLOAT else pa.int64())
                     for f in BLAST_FIELDS}
            tbl = pacsv.read_csv(
                path,
                read_options=pacsv.ReadOptions(column_names=BLAST_FIELDS, autogenerate_column_names=False),
                parse_options=pacsv.ParseOptions(delimiter="\t", quote_char='"', double_quote=True,
                                                 newlines_in_values=False),
                convert_options=pacsv.ConvertOptions(column_types=types, strings_can_be_null=False,
                                                     null_values=[], quoted_strings_can_be_null=False))
            if tbl.num_rows == 0:
                return hits_from_columns(*([[]] * 10))
            cols = {f: (tbl[f] if f in _BLAST_STR else tbl[f].to_numpy()) for f in want}
            ok = not pc.any(pc.equal(tbl["sstrand"], "")).as_py()
        except SystemExit:
            raise
        except Exception:
            cols, ok = None, False
    if cols is None or not ok:
        with try_open(path) as fh:
            text = fh.read()
        if not text.strip():
            return hits_from_columns(*([[]] * 10))
    if cols is None:
        dtypes = {f: (str if f in _BLAST_STR else np.float64 if f in _BLAST_FLOAT else np.int64)
                  for f in BLAST_FIELDS}
        try:
            df = pd.read_csv(io.StringIO(text), sep="\t", header=None, names=BLAST_FIELDS,
                             dtype=dtypes, float_precision="round_trip", na_filter=False,
                             quoting=csv.QUOTE_MINIMAL, index_col=False)
            ok = not (df["sstrand"] == "").any()
            cols = {f: df[f].to_numpy(dtype=object if f in _BLAST_STR else None) for f in want}
        except Exception:
            ok = False
    if not ok:
        for line in text.split("\n"):
            if line and line.count("\t") != len(BLAST_FIELDS) - 1:
                die("inconsistent blast row: {}".format(str(line.split("\t"))))   # UT:208-209
        die("unparseable blast file:", path)
    return hits_from_columns(*(cols[f] for f in want))


def _read_bytes(path):
    with try_open(path) as fh:
        return fh.buffer.read() if hasattr(fh, "buffer") else fh.read().encode()


def _gpu_parse_blast(path, device, genes=None):
    """The blastout parsed on the GPU (None: the CPU reader must take the file).  `genes` = (min_overlap, min_gene_length,
    min_scov): gene calls over the parsed columns, returned as (HitTable, genes).  The parser stays open with the hit
    columns on the device (HitTable.resident): the caller closes it (close_resident) once it has scored.  A BGZF blastout
    is inflated on the device (its compressed bytes cross PCIe, not the text); other compressed files are inflated on
    the host.  A BGZF member that fails validation on the device sends the file to the CPU reader, which raises the error
    Python's gzip raises on it."""
    from . import compressed, gpu_parse
    kind, members = compressed.classify(path)
    if kind == compressed.BGZF:
        with open(path, "rb") as fh:
            comp = fh.read()
    else:
        text = _read_bytes(path)
    parser = gpu_parse.BlastParser(device)
    try:
        if kind == compressed.BGZF:
            try:
                hits = parser.parse_bgzf(comp, members)
                say("  blastout: BGZF, {:,} members inflated on cuda:{}".format(len(members), device))
            except gpu_parse.InflateError as exc:
                say("  blastout: BGZF member {} failed validation on cuda:{}; reading the file on the host".format(
                    exc.member, device))
                hits = None
        else:
            hits = parser.parse(text)
        calls = parser.call_genes(*genes) if genes is not None and hits is not None else None
    except BaseException:
        parser.close()
        raise
    if hits is None:
        parser.close()
    else:
        hits.parse_times = parser.times
    return hits if genes is None else (hits, calls)


def close_resident(hits):
    """Close the GPU parser that holds the device columns of `hits`, if any."""
    r = getattr(hits, "resident", None)
    if r is not None:
        r.parser.close()


def read_blast_hits_and_genes(path, min_overlap, min_gene_length, min_scov, device=0, cpu_parse=False):
    """read_blast_hits plus the waafle_genecaller gene calls of its contig blocks, from one read of the file:
    (HitTable, (block names, gene_off [n_blocks + 1], start, end, strand char codes)).  The GPU parser's columns stay on
    the device for the gene calls; a file it cannot reproduce (or `cpu_parse`) goes through the CPU reader and
    genecaller.call_genes over the host columns, on `device` all the same."""
    from . import genecaller
    if not cpu_parse:
        hits, genes = _gpu_parse_blast(path, device, (min_overlap, min_gene_length, min_scov))
        if hits is not None:
            return hits, (list(hits.block_names) if hits.block_names is not None else [],) + tuple(genes)
    hits = read_blast_hits(path)
    names, gene_off, start, end, strand, _ = genecaller.call_genes(hits, min_overlap, min_gene_length, min_scov, device)
    return hits, (names, gene_off, start, end, strand)


class LocusTable:
    """All loci of a GFF file, in file order."""

    def __init__(self, seqname, start, end, strand_str):
        self.seqname = np.asarray(seqname, dtype=object)
        self.start = np.asarray(start, dtype=np.int32)
        self.end = np.asarray(end, dtype=np.int32)
        self.strand_str = np.asarray(strand_str, dtype=object)
        self.strand = np.array([ord(s) if len(s) == 1 else ord("?") for s in self.strand_str],
                               dtype=np.int8)

    @classmethod
    def from_blocks(cls, names, off, start, end, strand):
        """Loci as runs of one seqname: rows off[b] .. off[b + 1] belong to names[b]; `strand` holds char codes.  The
        gene calls of a blastout (names = its contig blocks) give the table read_gff_loci reads from their GFF."""
        lt = cls.__new__(cls)
        counts = np.diff(np.asarray(off, dtype=np.int64))
        lt.seqname = np.repeat(np.array(names, dtype=object), counts) if len(names) else np.zeros(0, dtype=object)
        lt.start = np.ascontiguousarray(start, dtype=np.int32)
        lt.end = np.ascontiguousarray(end, dtype=np.int32)
        lt.strand = np.ascontiguousarray(strand, dtype=np.int8)
        lt.strand_str = lt.strand.view("S1").astype(str).astype(object)
        return lt

    def __len__(self):
        return len(self.start)

    def code(self, j):
        """`start:end:strand` (UT:317)."""
        return "{}:{}:{}".format(int(self.start[j]), int(self.end[j]), self.strand_str[j])


def read_gff_loci(path, device=None):
    """Parse a GFF (waafle_genecaller or Prodigal style); `#` rows are skipped (UT:345-346).  With `device` (a CUDA device
    index) the rows are parsed on the GPU (gpu_parse.BlastParser.parse_gff); files it cannot reproduce fall through to the
    CPU reader below, which has the reference's error behaviour."""
    if device is not None:
        from . import gpu_parse
        text = _read_bytes(path)
        parser = gpu_parse.BlastParser(device)
        try:
            loci = parser.parse_gff(text)
        finally:
            parser.close()
        if loci is not None:
            loci.parse_times = parser.times
            return loci
    with try_open(path) as fh:
        lines = [ln for ln in fh.read().split("\n") if ln and ln[0] != "#"]
    for ln in lines:
        if ln.count("\t") != len(GFF_FIELDS) - 1:
            die("Bad GFF row:", ln.split("\t"))   # UT:302-303
    if not lines:
        return LocusTable([], [], [], [])
    df = pd.read_csv(io.StringIO("\n".join(lines)), sep="\t", header=None, names=GFF_FIELDS,
                     dtype=str, na_filter=False, quoting=csv.QUOTE_NONE, index_col=False)
    return LocusTable(df["seqname"].to_numpy(dtype=object), df["start"].astype(np.int64),
                      df["end"].astype(np.int64), df["strand"].to_numpy(dtype=object))
