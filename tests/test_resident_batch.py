"""CPU: the host half of the device-built scoring batch.  `packing.map_contigs` gives the arrays the packer built before
it was factored out, and `ResidentBatch.hit_row` / `slice` agree with the host `Batch`."""
import copy
import os

import numpy as np

import helpers
from waafle_b200 import packing, parsers, synth, taxonomy, utils


def _old_mapping(contig_lengths, loci, hits):
    """The contig / locus / hit mapping as `pack` computed it before map_contigs (two stable argsorts)."""
    names = list(contig_lengths)
    index = {n: i for i, n in enumerate(names)}
    n = len(names)
    lc = np.fromiter((index.get(x, -1) for x in loci.seqname), dtype=np.int64, count=len(loci.seqname))
    lrow = np.nonzero(lc >= 0)[0]
    lrow = lrow[np.argsort(lc[lrow], kind="stable")]
    locus_off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(lc[lrow], minlength=n), out=locus_off[1:])
    if hits.block_starts is not None and len(hits):
        bcid = np.fromiter((index.get(x, -1) for x in hits.block_names), dtype=np.int64, count=len(hits.block_names))
        hc = np.repeat(bcid, np.diff(np.r_[hits.block_starts, len(hits)]))
    else:
        hc = np.fromiter((index.get(x, -1) for x in hits.qseqid), dtype=np.int64, count=len(hits.qseqid))
    hrow = np.nonzero(hc >= 0)[0]
    hrow = hrow[np.argsort(hc[hrow], kind="stable")]
    hit_off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(hc[hrow], minlength=n), out=hit_off[1:])
    return locus_off, lrow, hit_off, hrow


def _with_blocks(hits):
    """A copy of the HitTable with the GPU parser's run-length view of the query names."""
    hits = copy.copy(hits)
    q = hits.qseqid
    starts = np.flatnonzero(np.r_[True, q[1:] != q[:-1]]) if len(q) else np.zeros(0, np.int64)
    hits.block_starts, hits.block_names = starts.astype(np.int64), [q[s] for s in starts]
    return hits


class _FakeParser:
    is_open, generation = True, 1


def _inputs(tmp_path, kind):
    os.makedirs(str(tmp_path), exist_ok=True)
    if kind == "demo":
        files = helpers.demo_files(tmp_path)
    else:
        data = synth.generate_config(kind, n_contigs=120, seed=17, annotations=kind == "cfg5")
        files = data.write_files(str(tmp_path), kind)
    lengths = utils.read_contig_lengths(files["contigs"])
    # a FASTA order other than the blastout's, contigs the blastout lacks and blastout contigs the FASTA lacks
    names = list(lengths)
    rng = np.random.default_rng(3)
    keep = [names[i] for i in rng.permutation(len(names))[: len(names) - 3]] + ["extra_a", "extra_b"]
    lengths = {nm: lengths.get(nm, 1000) for nm in keep}
    loci = parsers.read_gff_loci(files["gff"])
    hits = parsers.read_blast_hits(files["blastout"])
    tax = taxonomy.Taxonomy(files["taxonomy"]).build(hits.distinct_taxa())
    return lengths, loci, hits, tax


def test_map_contigs_equals_the_old_mapping(tmp_path):
    for kind in ("demo", "cfg2", "cfg5"):
        lengths, loci, hits, tax = _inputs(tmp_path / kind, kind)
        for table in (hits, _with_blocks(hits)):
            names, locus_off, lrow, hit_off, hit_src, hc = packing.map_contigs(lengths, loci, table)
            o_locus_off, o_lrow, o_hit_off, o_hrow = _old_mapping(lengths, loci, table)
            assert names == list(lengths)
            for a, b in ((locus_off, o_locus_off), (lrow, o_lrow), (hit_off, o_hit_off)):
                assert np.array_equal(a, b), kind
            hrow = packing.block_rows(hit_off, hit_src) if hc is None else None
            if hrow is not None:
                assert np.array_equal(hrow, o_hrow), kind
            batch = packing.pack(lengths, loci, table, tax)
            assert np.array_equal(np.sort(batch.hit_row), np.sort(o_hrow))


def test_resident_batch_hit_row_and_slice_agree_with_batch(tmp_path):
    for kind in ("demo", "cfg2", "cfg5"):
        lengths, loci, hits, tax = _inputs(tmp_path / kind, kind)
        hits = _with_blocks(hits)
        from waafle_b200 import gpu_parse
        hits.resident = gpu_parse.ResidentParse(_FakeParser(), 1, np.arange(len(hits.taxon_names)), None)
        host = packing.pack(lengths, loci, hits, tax)
        res = packing.pack_resident(lengths, loci, hits, tax)
        assert res.slot_node[: len(hits.taxon_names)].tolist() == [tax.index[t] for t in hits.taxon_names]
        for c0, c1 in ((0, res.n_contigs), (0, 1), (5, 40), (res.n_contigs - 7, res.n_contigs)):
            a, b = host.slice(c0, c1), res.slice(c0, c1)
            assert a.n_contigs == b.n_contigs and a.n_hits == b.n_hits and a.n_loci == b.n_loci
            for k in ("hit_off", "locus_off", "locus_start", "locus_end", "locus_strand", "contig_lengths", "locus_row"):
                assert np.array_equal(getattr(a, k), getattr(b, k)), (kind, k)
            assert a.contig_names == b.contig_names
            if host.hit_sysmask is not None:   # annotations: file order, the rows are the same
                assert np.array_equal(a.hit_row, b.hit_row), kind
            else:   # sorted per contig on the host: the same rows in another order
                for c in range(a.n_contigs):
                    lo, hi = a.hit_off[c], a.hit_off[c + 1]
                    assert np.array_equal(np.sort(a.hit_row[lo:hi]), b.hit_row[lo:hi]), kind


def test_pack_resident_needs_a_live_parse(tmp_path):
    lengths, loci, hits, tax = _inputs(tmp_path, "demo")
    hits = _with_blocks(hits)
    from waafle_b200 import gpu_parse
    parser = _FakeParser()
    hits.resident = gpu_parse.ResidentParse(parser, 0, np.arange(len(hits.taxon_names)), None)
    assert gpu_parse.live_resident(hits) is None   # the parser has parsed again since
    try:
        packing.pack_resident(lengths, loci, hits, tax)
    except ValueError:
        pass
    else:
        raise AssertionError("pack_resident accepted a stale parse")
