"""CSR/SoA packing of contigs, loci and hits: the host side of the drop-in boundary.

The reference keeps one `Contig` object per FASTA record holding lists of `Locus`
and `Hit` objects (waafle/waafle_orgscorer.py:908-925, 943-953).  Here the same
information is laid out as the flat arrays of `wfl_batch` (include/waafle_b200.h):
contigs in FASTA order, loci in GFF order and hits in blastout order inside each
contig (the reference's iteration orders: UT:255-270, UT:341-355).
"""

from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from .utils import die, say

_ARRAYS = ["hit_off", "locus_off", "hit_qstart", "hit_qend", "hit_taxon", "hit_score",
           "hit_scov", "hit_strand", "hit_sysmask", "locus_start", "locus_end", "locus_strand"]


@dataclass
class Batch:
    hit_off: np.ndarray        # int64 [n+1]
    locus_off: np.ndarray      # int64 [n+1]
    hit_qstart: np.ndarray     # int32 [H]
    hit_qend: np.ndarray       # int32 [H]
    hit_taxon: np.ndarray      # int32 [H]  node index (taxonomy.Taxonomy.index)
    hit_score: np.ndarray      # float64 [H] waafle_score
    hit_scov: np.ndarray       # float64 [H] scov_modified
    hit_strand: np.ndarray     # int8 [H]
    locus_start: np.ndarray    # int32 [L]
    locus_end: np.ndarray      # int32 [L]
    locus_strand: np.ndarray   # int8 [L]
    hit_sysmask: Optional[np.ndarray] = None   # uint32 [H]
    # host-only side tables (never shipped to the device)
    contig_names: list = field(default_factory=list)
    contig_lengths: Optional[np.ndarray] = None
    hit_row: Optional[np.ndarray] = None       # index of each packed hit in the HitTable
    locus_row: Optional[np.ndarray] = None     # index of each packed locus in the LocusTable

    @property
    def n_contigs(self):
        return len(self.hit_off) - 1

    @property
    def n_hits(self):
        return int(self.hit_off[-1])

    @property
    def n_loci(self):
        return int(self.locus_off[-1])

    def arrays(self):
        """Dict of the device-facing arrays (what the C ABI and the oracle consume)."""
        return {k: getattr(self, k) for k in _ARRAYS if getattr(self, k) is not None}

    def slice(self, c0, c1):
        """Contigs [c0, c1) as an independent batch with rebased offsets."""
        h0, h1 = int(self.hit_off[c0]), int(self.hit_off[c1])
        l0, l1 = int(self.locus_off[c0]), int(self.locus_off[c1])
        cut = lambda a, lo, hi: None if a is None else a[lo:hi]
        return Batch(
            hit_off=self.hit_off[c0:c1 + 1] - h0, locus_off=self.locus_off[c0:c1 + 1] - l0,
            hit_qstart=self.hit_qstart[h0:h1], hit_qend=self.hit_qend[h0:h1],
            hit_taxon=self.hit_taxon[h0:h1], hit_score=self.hit_score[h0:h1],
            hit_scov=self.hit_scov[h0:h1], hit_strand=self.hit_strand[h0:h1],
            locus_start=self.locus_start[l0:l1], locus_end=self.locus_end[l0:l1],
            locus_strand=self.locus_strand[l0:l1], hit_sysmask=cut(self.hit_sysmask, h0, h1),
            contig_names=self.contig_names[c0:c1],
            contig_lengths=cut(self.contig_lengths, c0, c1),
            hit_row=cut(self.hit_row, h0, h1), locus_row=cut(self.locus_row, l0, l1))

    def sort_hits(self):
        """The same batch with every contig's hits in the order the fused fast-path kernel visits them at the first
        taxonomy level: by (taxon index, descending waafle_score) -- the kernel then only CHECKS the order instead of
        sorting in shared memory.  Semantically transparent: envelopes are order-free.  One stable integer sort of a
        composite key  contig | taxon | quantised score  (15 M hits/s; np.lexsort on the four columns does 1 M hits/s);
        scores that collide in the quantisation may stay in file order, which the kernel detects and repairs per contig.
        With annotation systems the hits stay in FILE order: the annotation tie-break "last hit in file order" (OS:389) is
        "largest index among equal scores" there, and the kernel sorts by clade itself."""
        if self.hit_sysmask is not None or self.n_hits == 0:
            return self
        n = self.n_contigs
        contig = np.repeat(np.arange(n, dtype=np.int64), np.diff(self.hit_off))
        bits_c = max(1, int(n - 1).bit_length())
        bits_t = max(1, int(self.hit_taxon.max(initial=0)).bit_length())
        bits_s = 63 - bits_c - bits_t
        score = np.nan_to_num(self.hit_score, nan=0.0, posinf=0.0, neginf=0.0)
        smax = float(score.max(initial=0.0))
        if bits_s >= 20 and smax > 0.0 and int(self.hit_taxon.min(initial=0)) >= 0:
            q = ((smax - np.clip(score, 0.0, smax)) * (float((1 << bits_s) - 1) / smax)).astype(np.int64)
            key = (contig << (bits_t + bits_s)) | (self.hit_taxon.astype(np.int64) << bits_s) | q
            order = np.argsort(key, kind="stable")
        else:
            order = np.lexsort((np.arange(len(contig)), -self.hit_score, self.hit_taxon, contig))
        take = lambda a: None if a is None else np.ascontiguousarray(a[order])
        return Batch(
            hit_off=self.hit_off, locus_off=self.locus_off,
            hit_qstart=take(self.hit_qstart), hit_qend=take(self.hit_qend), hit_taxon=take(self.hit_taxon),
            hit_score=take(self.hit_score), hit_scov=take(self.hit_scov), hit_strand=take(self.hit_strand),
            locus_start=self.locus_start, locus_end=self.locus_end, locus_strand=self.locus_strand,
            hit_sysmask=take(self.hit_sysmask), contig_names=self.contig_names, contig_lengths=self.contig_lengths,
            hit_row=take(self.hit_row), locus_row=self.locus_row)

    def can_pack(self, n_nodes, n_systems=0):
        """True if the compact wire format (wfl_packed_batch) can carry this batch."""
        hi = max(int(self.hit_qstart.max(initial=0)), int(self.hit_qend.max(initial=0)))
        lo = min(int(self.hit_qstart.min(initial=0)), int(self.hit_qend.min(initial=0)))
        return n_nodes <= 16384 and n_systems <= 8 and lo >= 0 and hi <= 65535

    def to_packed(self, min_scov):
        """The device-facing arrays in the compact wire format (14 B/hit instead of 29): the scov filter of
        waafle_orgscorer.py:362 is applied here (one bit), the strand is one bit, taxon and coordinates 16-bit."""
        tax16 = (self.hit_taxon.astype(np.uint16)
                 | np.where(self.hit_strand == ord("-"), np.uint16(0x4000), np.uint16(0))
                 | np.where(self.hit_scov >= min_scov, np.uint16(0x8000), np.uint16(0))).astype(np.uint16)
        out = dict(hit_off=self.hit_off, locus_off=self.locus_off,
                   hit_qstart16=self.hit_qstart.astype(np.uint16), hit_qend16=self.hit_qend.astype(np.uint16),
                   hit_tax16=tax16, hit_score=self.hit_score, locus_start=self.locus_start,
                   locus_end=self.locus_end, locus_strand=self.locus_strand)
        if self.hit_sysmask is not None:
            out["hit_sysmask8"] = self.hit_sysmask.astype(np.uint8)
        return out

    def algorithmic_bytes(self, n_systems=0):
        """SURVEY.md 8(d): 29 B/hit + 9 B/locus + 16 B/contig in, 40 + G(1+4S) B/contig out."""
        return (29 * self.n_hits + 9 * self.n_loci + 16 * self.n_contigs
                + 40 * self.n_contigs + self.n_loci * (1 + 4 * n_systems))


def concat_batches(parts):
    """Concatenate batches (contigs of parts[0], then parts[1], ...) with rebased offsets."""
    def cat(name):
        arrs = [getattr(p, name) for p in parts]
        return None if any(a is None for a in arrs) else np.concatenate(arrs)

    def cat_off(name, total_name):
        out, base = [np.zeros(1, np.int64)], 0
        for p in parts:
            o = getattr(p, name)
            out.append(o[1:] + base)
            base += int(o[-1])
        return np.concatenate(out)

    names = []
    for p in parts:
        names += list(p.contig_names)
    return Batch(
        hit_off=cat_off("hit_off", "n_hits"), locus_off=cat_off("locus_off", "n_loci"),
        hit_qstart=cat("hit_qstart"), hit_qend=cat("hit_qend"), hit_taxon=cat("hit_taxon"),
        hit_score=cat("hit_score"), hit_scov=cat("hit_scov"), hit_strand=cat("hit_strand"),
        locus_start=cat("locus_start"), locus_end=cat("locus_end"), locus_strand=cat("locus_strand"),
        hit_sysmask=cat("hit_sysmask"), contig_names=names, contig_lengths=cat("contig_lengths"))


def tiled_slice(base, c0, c1):
    """Contigs [c0, c1) of the infinite tiling base, base, base, ... (synthetic weak / strong scaling workloads)."""
    n = base.n_contigs
    parts = []
    c = c0
    while c < c1:
        lo = c % n
        hi = min(n, lo + (c1 - c))
        parts.append(base.slice(lo, hi))
        c += hi - lo
    return concat_batches(parts) if len(parts) != 1 else parts[0]


def _group(names, index, what, codes=None, code_names=None):
    """Map row -> contig index; unknown contigs are warned about and dropped like OS:921-923.
    `codes` / `code_names`: optional dictionary encoding of `names` (one lookup per distinct name)."""
    if codes is not None and len(codes) == len(names):
        lut = np.fromiter((index.get(n, -1) for n in code_names), dtype=np.int64, count=len(code_names))
        cid = lut[codes] if len(codes) else np.zeros(0, dtype=np.int64)
    else:
        cid = np.fromiter((index.get(n, -1) for n in names), dtype=np.int64, count=len(names))
    if len(cid):
        starts = np.r_[True, names[1:] != names[:-1]]
        for n in names[starts & (cid < 0)]:
            say("  Unknown contig in <{}> file".format(what), n)
    return cid


def block_rows(hit_off, hit_src):
    """Row of every packed hit in the HitTable when contig c holds rows [hit_src[c], hit_src[c] + its hit count)."""
    counts = np.diff(hit_off)
    n_hits = int(hit_off[-1])
    return np.repeat(np.asarray(hit_src, np.int64) - hit_off[:-1], counts) + np.arange(n_hits, dtype=np.int64)


def map_contigs(contig_lengths, loci, hits):
    """Where the contigs of `pack` find their loci and hits: (names, locus_off, locus_row, hit_off, hit_src, hit_contig).
    Contigs in FASTA order; unknown contigs are warned about and dropped (OS:921-923); a blastout that is not grouped
    by query dies (UT:255-258).  Loci: locus_row[locus_off[c]:locus_off[c + 1]] are contig c's rows of `loci`.  Hits,
    for a HitTable with block_starts (every contig is one block of rows): hit_src[c] = first row of contig c's block
    (0 without hits), hit_contig = None; otherwise hit_src = None and hit_contig = the contig of every row (-1:
    unknown)."""
    names = list(contig_lengths)
    index = {n: i for i, n in enumerate(names)}
    n = len(names)

    lc = _group(loci.seqname, index, "gff")
    lrow = np.nonzero(lc >= 0)[0]
    lrow = lrow[np.argsort(lc[lrow], kind="stable")]
    locus_off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(lc[lrow], minlength=n), out=locus_off[1:])

    hit_off = np.zeros(n + 1, dtype=np.int64)
    if getattr(hits, "block_starts", None) is not None and len(hits):
        # run-length coded query names (GPU parser): one lookup per block, no per-row objects
        bcid = np.fromiter((index.get(nm, -1) for nm in hits.block_names), dtype=np.int64, count=len(hits.block_names))
        for nm in np.array(hits.block_names, dtype=object)[bcid < 0]:
            say("  Unknown contig in <{}> file".format("blastout"), nm)
        known = bcid >= 0
        if len(np.unique(bcid[known])) != int(known.sum()):   # the reference assumes the blastout is grouped by query (UT:255-258)
            die("blastout is not grouped by query sequence")
        starts = np.asarray(hits.block_starts, dtype=np.int64)
        lens = np.diff(np.r_[starts, len(hits)])
        counts = np.zeros(n, dtype=np.int64)
        counts[bcid[known]] = lens[known]
        np.cumsum(counts, out=hit_off[1:])
        hit_src = np.zeros(n, dtype=np.int64)
        hit_src[bcid[known]] = starts[known]
        return names, locus_off, lrow, hit_off, hit_src, None
    hc = _group(hits.qseqid, index, "blastout", getattr(hits, "qseqid_codes", None), getattr(hits, "qseqid_names", None))
    if len(hc):
        # the reference assumes the blastout is grouped by query (UT:255-258)
        starts = np.r_[True, hits.qseqid[1:] != hits.qseqid[:-1]]
        blocks = hc[starts]
        blocks = blocks[blocks >= 0]
        if len(np.unique(blocks)) != len(blocks):
            die("blastout is not grouped by query sequence")
    np.cumsum(np.bincount(hc[hc >= 0], minlength=n), out=hit_off[1:])
    return names, locus_off, lrow, hit_off, None, hc


def pack(contig_lengths, loci, hits, taxonomy):
    """Pack parsed inputs. `taxonomy` must already be built with the hit taxa as extra names."""
    names, locus_off, lrow, hit_off, hit_src, hc = map_contigs(contig_lengths, loci, hits)
    if hc is None:
        hrow = block_rows(hit_off, hit_src)
    else:
        hrow = np.nonzero(hc >= 0)[0]
        hrow = hrow[np.argsort(hc[hrow], kind="stable")]

    if getattr(hits, "taxon_codes", None) is not None:
        tlut = np.fromiter((taxonomy.index[t] for t in hits.taxon_names), dtype=np.int32, count=len(hits.taxon_names))
        taxon = tlut[hits.taxon_codes[hrow]] if len(hrow) else np.zeros(0, dtype=np.int32)
    else:
        taxon = np.fromiter((taxonomy.index[t] for t in hits.taxon[hrow]), dtype=np.int32,
                            count=len(hrow))
    return Batch(
        hit_off=hit_off, locus_off=locus_off,
        hit_qstart=np.ascontiguousarray(hits.qstart[hrow]),
        hit_qend=np.ascontiguousarray(hits.qend[hrow]),
        hit_taxon=taxon,
        hit_score=np.ascontiguousarray(hits.score[hrow]),
        hit_scov=np.ascontiguousarray(hits.scov_modified[hrow]),
        hit_strand=np.ascontiguousarray(hits.strand[hrow]),
        hit_sysmask=None if hits.sysmask is None or not hits.systems
        else np.ascontiguousarray(hits.sysmask[hrow]),
        locus_start=np.ascontiguousarray(loci.start[lrow]),
        locus_end=np.ascontiguousarray(loci.end[lrow]),
        locus_strand=np.ascontiguousarray(loci.strand[lrow]),
        contig_names=names,
        contig_lengths=np.array([contig_lengths[k] for k in names], dtype=np.int64),
        hit_row=hrow, locus_row=lrow).sort_hits()


@dataclass
class ResidentBatch:
    """The batch `pack` would build, with its hit columns left in a GPU parser's device columns: Engine.score_batch builds
    them there (wfl_upload_parsed).  Carries the host-side fields the writer and the streamed runs read; contig c's hits
    are the parser rows [hit_src[c], hit_src[c] + its hit count)."""
    hit_off: np.ndarray        # int64 [n+1]
    locus_off: np.ndarray      # int64 [n+1]
    hit_src: np.ndarray        # int64 [n]  first parser row of every contig's block
    locus_start: np.ndarray    # int32 [L]
    locus_end: np.ndarray      # int32 [L]
    locus_strand: np.ndarray   # int8 [L]
    resident: object = None    # gpu_parse.ResidentParse of the hits
    slot_node: Optional[np.ndarray] = None   # int32 [2^20] distinct-taxon slot -> node index, -1 unused
    contig_names: list = field(default_factory=list)
    contig_lengths: Optional[np.ndarray] = None
    locus_row: Optional[np.ndarray] = None

    n_contigs = Batch.n_contigs
    n_hits = Batch.n_hits
    n_loci = Batch.n_loci

    @property
    def hit_row(self):
        """Index of each packed hit in the HitTable.  Only annotation winners read it, and with annotation systems the
        hits stay in file order, so this is exact wherever it is read."""
        return block_rows(self.hit_off, self.hit_src)

    def slice(self, c0, c1):
        """Contigs [c0, c1) as an independent batch with rebased offsets (the parser rows stay where they are)."""
        h0, l0, l1 = int(self.hit_off[c0]), int(self.locus_off[c0]), int(self.locus_off[c1])
        cut = lambda a, lo, hi: None if a is None else a[lo:hi]
        return ResidentBatch(
            hit_off=self.hit_off[c0:c1 + 1] - h0, locus_off=self.locus_off[c0:c1 + 1] - l0,
            hit_src=self.hit_src[c0:c1], locus_start=self.locus_start[l0:l1], locus_end=self.locus_end[l0:l1],
            locus_strand=self.locus_strand[l0:l1], resident=self.resident, slot_node=self.slot_node,
            contig_names=self.contig_names[c0:c1], contig_lengths=cut(self.contig_lengths, c0, c1),
            locus_row=cut(self.locus_row, l0, l1))


def pack_resident(contig_lengths, loci, hits, taxonomy):
    """`pack` for hits whose GPU parse is still live (gpu_parse.live_resident): the contig, block and locus mapping on the
    host, the hit columns left on the device.  `taxonomy` must already be built with the hit taxa as extra names."""
    from .gpu_parse import TAX_SLOTS, live_resident
    res = live_resident(hits)
    if res is None:
        raise ValueError("pack_resident: the hits carry no live GPU parse")
    names, locus_off, lrow, hit_off, hit_src, hc = map_contigs(contig_lengths, loci, hits)
    if hit_src is None:   # no rows (an empty blastout): nothing to locate
        hit_src = np.zeros(len(names), dtype=np.int64)
    slot_node = np.full(TAX_SLOTS, -1, np.int32)
    if len(res.taxon_slots):
        slot_node[res.taxon_slots] = np.fromiter((taxonomy.index[t] for t in hits.taxon_names), dtype=np.int32,
                                                 count=len(hits.taxon_names))
    return ResidentBatch(
        hit_off=hit_off, locus_off=locus_off, hit_src=hit_src,
        locus_start=np.ascontiguousarray(loci.start[lrow]), locus_end=np.ascontiguousarray(loci.end[lrow]),
        locus_strand=np.ascontiguousarray(loci.strand[lrow]), resident=res, slot_node=slot_node,
        contig_names=names, contig_lengths=np.array([contig_lengths[k] for k in names], dtype=np.int64),
        locus_row=lrow)
