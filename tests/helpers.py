"""Shared test helpers: oracle-vs-engine array comparison, golden IO."""

import gzip
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

EXACT_FIELDS = ["call", "direction", "lifts", "clade1", "clade2", "lca", "best1", "best2",
                "synteny", "locus_flags", "ann_winner", "member_off", "n_members_a", "members",
                "call_counts", "call_index"]


def compare_results(ref, got, score_rtol=0.0):
    """All integer/byte outputs bit-exact; crit/rank bit-exact (score_rtol=0) or within rtol."""
    diffs = []
    for k in EXACT_FIELDS:
        a, b = np.asarray(ref[k]), np.asarray(got[k])
        if a.shape != b.shape:
            diffs.append((k, "shape", a.shape, b.shape))
        elif not np.array_equal(a, b):
            bad = np.nonzero(a.reshape(len(a), -1) != b.reshape(len(b), -1))[0]
            diffs.append((k, "first_bad", int(bad[0]), a[bad[0]].tolist(), b[bad[0]].tolist(),
                          "n_bad", len(np.unique(bad))))
    for k in ("crit", "rank"):
        a, b = np.asarray(ref[k]), np.asarray(got[k])
        if score_rtol == 0.0:
            ok = a.view(np.int64) == b.view(np.int64)
        else:
            ok = np.abs(a - b) <= score_rtol * np.maximum(np.abs(a), np.abs(b))
        if not ok.all():
            i = int(np.nonzero(~ok)[0][0])
            diffs.append((k, "first_bad", i, float(a[i]).hex(), float(b[i]).hex(),
                          "n_bad", int((~ok).sum())))
    return diffs


def near_print_edge(x, tol=1e-11):
    """True if x lies within `tol` of a value that prints differently on either side at 4 decimals (x.xxxx5)."""
    y = float(x) * 1e4
    return abs(y - np.floor(y) - 0.5) <= tol * 1e4


def compare_printed(ref, got):
    """crit / rank of every contig the reference classifies, as the TSV writer prints them (4 decimals)."""
    from waafle_b200.utils import format_field
    diffs = []
    for c in np.nonzero(np.asarray(ref["call"]) != 0)[0]:
        for k in ("crit", "rank"):
            a, b = format_field(float(ref[k][c])), format_field(float(got[k][c]))
            if a != b:
                diffs.append((k, int(c), a, b, float(ref[k][c]).hex(), float(got[k][c]).hex()))
    return diffs


def load_json(name):
    path = os.path.join(GOLDEN, name)
    if path.endswith(".gz"):
        with gzip.open(path, "rt") as fh:
            return json.load(fh)
    with open(path) as fh:
        return json.load(fh)


# ---------------------------------------------------------------------------------------------
# inputs: demo fixtures, seeded synthetic cases, hand-built adversarial batches
# ---------------------------------------------------------------------------------------------

def demo_files(tmpdir, prodigal=False):
    """Paths of the demo inputs; the FASTA is rebuilt from the stored contig lengths."""
    d = os.path.join(GOLDEN, "demo")
    fna = os.path.join(str(tmpdir), "demo_contigs.fna")
    if not os.path.exists(fna):
        with open(os.path.join(d, "demo_contigs.lengths.tsv")) as fh, open(fna, "w") as out:
            for line in fh:
                name, length = line.split("\t")
                out.write(">{}\n{}\n".format(name, "N" * int(length)))
    return dict(contigs=fna, blastout=os.path.join(d, "demo_contigs.blastout"),
                gff=os.path.join(d, "demo_contigs.prodigal.gff" if prodigal else "demo_contigs.gff"),
                taxonomy=os.path.join(d, "demo_taxonomy.tsv"))


def frontend_load(files):
    from waafle_b200 import packing, parsers, taxonomy, utils
    hits = parsers.read_blast_hits(files["blastout"])
    loci = parsers.read_gff_loci(files["gff"])
    tax = taxonomy.Taxonomy(files["taxonomy"]).build(set(hits.taxon))
    batch = packing.pack(utils.read_contig_lengths(files["contigs"]), loci, hits, tax)
    return batch, loci, hits, tax


def params_for(flags, n_systems=0):
    """Reference-CLI style flag dict (argparse attribute names) -> OrgscorerParams."""
    from oracle.reference_harness import make_args
    from waafle_b200.params import OrgscorerParams
    return OrgscorerParams.from_args(make_args(**flags), n_systems)


def decode_golden(records):
    out = {}
    for name, r in records.items():
        r = dict(r)
        for k in ("crit", "rank"):
            if k in r:
                r[k] = float.fromhex(r[k])
        r.setdefault("gene_scores0", {})
        out[name] = r
    return out


def synth_case(case):
    from waafle_b200 import synth
    over = {k: tuple(v) if isinstance(v, list) else v for k, v in case["over"].items()}
    return synth.generate_config(case["config"], n_contigs=case["n_contigs"], seed=case["seed"], **over)


def batch_checksum(batch):
    import hashlib
    h = hashlib.sha256()
    for k in sorted(batch.arrays()):
        h.update(batch.arrays()[k].tobytes())
    return h.hexdigest()


def make_batch(contigs, edges, extra_taxa=()):
    """Hand-built batch.  contigs: list of dict(loci=[(start, end, strand_char)],
    hits=[(qstart, qend, taxon_name, score, scov, strand_char[, sysmask])]).
    edges: [(clade, parent)] taxonomy rows.  Returns (Batch, Taxonomy)."""
    from waafle_b200.packing import Batch
    from waafle_b200.taxonomy import Taxonomy
    taxa = {h[2] for c in contigs for h in c.get("hits", [])} | set(extra_taxa)
    tax = Taxonomy(edges=[list(e) for e in edges]).build(taxa)
    hit_off, locus_off = [0], [0]
    H = {k: [] for k in ("q1", "q2", "tx", "sc", "cv", "st", "sm")}
    L = {k: [] for k in ("s", "e", "st")}
    for c in contigs:
        for l in c.get("loci", []):
            L["s"].append(l[0]); L["e"].append(l[1]); L["st"].append(ord(l[2]))
        for h in c.get("hits", []):
            H["q1"].append(h[0]); H["q2"].append(h[1]); H["tx"].append(tax.index[h[2]])
            H["sc"].append(h[3]); H["cv"].append(h[4]); H["st"].append(ord(h[5]))
            H["sm"].append(h[6] if len(h) > 6 else 1)
        hit_off.append(len(H["q1"])); locus_off.append(len(L["s"]))
    b = Batch(
        hit_off=np.array(hit_off, np.int64), locus_off=np.array(locus_off, np.int64),
        hit_qstart=np.array(H["q1"], np.int32), hit_qend=np.array(H["q2"], np.int32),
        hit_taxon=np.array(H["tx"], np.int32), hit_score=np.array(H["sc"], np.float64),
        hit_scov=np.array(H["cv"], np.float64), hit_strand=np.array(H["st"], np.int8),
        locus_start=np.array(L["s"], np.int32), locus_end=np.array(L["e"], np.int32),
        locus_strand=np.array(L["st"], np.int8), hit_sysmask=np.array(H["sm"], np.uint32),
        contig_names=["c{:05d}".format(i) for i in range(len(contigs))],
        contig_lengths=np.array([c.get("length", 100000) for c in contigs], np.int64))
    return b, tax


TAX8 = [("k__B", "r__Root"), ("p__P1", "k__B"), ("p__P2", "k__B"), ("c__C1", "p__P1"), ("c__C2", "p__P2"),
        ("o__O1", "c__C1"), ("o__O2", "c__C2"), ("f__F1", "o__O1"), ("f__F2", "o__O2"),
        ("g__G1", "f__F1"), ("g__G2", "f__F1"), ("g__G3", "f__F2"),
        ("s__A", "g__G1"), ("s__B", "g__G1"), ("s__C", "g__G1"), ("s__D", "g__G2"), ("s__E", "g__G2"),
        ("s__F", "g__G3"), ("s__G", "g__G3"), ("t__A1", "s__A"), ("t__A2", "s__A")]


def adversarial_batches():
    """Named (batch, taxonomy) pairs exercising the edge cases SURVEY.md 8(d) lists."""
    out = {}
    # 1. knife edge: a gene fully covered at exactly 0.8 / 0.5 for every gene length 200..3000:
    #    np.mean of n copies of 0.8 is below 0.8 for most n (numpy pairwise rounding)
    cs = []
    for n in list(range(200, 460)) + list(range(460, 3001, 37)):
        for v in (0.8, 0.5, 0.1 + 0.7, 1.0):
            cs.append(dict(loci=[(1, n, "+"), (n + 50, 2 * n + 49, "-")],
                           hits=[(1, n, "s__A", v, 1.0, "+"), (n + 50, 2 * n + 49, "s__D", 1.0, 1.0, "+"),
                                 (3, n - 2, "s__B", 0.3, 0.9, "-")]))
    out["knife_edge"] = make_batch(cs, TAX8)
    # 2. exact rank ties with dyadic scores: three species at rank 0.875 on two 1000-bp genes
    cs = []
    for perm in (("s__A", "s__B", "s__C"), ("s__C", "s__A", "s__B"), ("s__D", "s__E", "s__F")):
        hits = []
        for sp, (v1, v2) in zip(perm, ((0.75, 1.0), (0.875, 0.875), (1.0, 0.75))):
            hits += [(1, 1000, sp, v1, 1.0, "+"), (1101, 2100, sp, v2, 1.0, "+")]
        cs.append(dict(loci=[(1, 1000, "+"), (1101, 2100, "+")], hits=hits))
    # two-clade ties: A covers gene1 only, {B, C} tie on gene2
    cs.append(dict(loci=[(1, 1000, "+"), (1101, 2100, "+"), (2201, 3200, "+")],
                   hits=[(1, 1000, "s__A", 1.0, 1.0, "+"), (2201, 3200, "s__A", 1.0, 1.0, "+"),
                         (1101, 2100, "s__F", 0.875, 1.0, "+"), (1101, 2100, "s__G", 0.875, 1.0, "+"),
                         (1101, 2100, "s__D", 0.875, 1.0, "+")]))
    out["ties"] = make_batch(cs, TAX8)
    # 3. multi-word gene masks: G in {63, 64, 65, 128, 129, 200}, LGT island in the middle
    cs = []
    for G in (63, 64, 65, 128, 129, 200):
        loci = [(1 + 400 * i, 300 + 400 * i, "+") for i in range(G)]
        hits = []
        for i in range(G):
            sp = "s__F" if G // 2 - 1 <= i <= G // 2 + 1 else "s__A"
            hits.append((1 + 400 * i, 300 + 400 * i, sp, 0.95, 1.0, "+"))
            if i % 7 == 0:
                hits.append((1 + 400 * i, 300 + 400 * i, "s__B", 0.6, 0.8, "-"))
            if i % 11 == 0:
                hits.append((11 + 400 * i, 290 + 400 * i, "s__G", 0.9, 0.9, "-"))
        cs.append(dict(loci=loci, hits=hits))
    out["multiword"] = make_batch(cs, TAX8)
    # 4. odd inputs: unsorted / reversed loci, reversed hit coordinates, overlapping loci, hits on
    #    several loci, unlisted taxa, "Unknown" as a hit taxon, scov > 1, failing scov, short loci,
    #    contigs without hits / without loci / with nothing
    cs = [
        dict(loci=[(2500, 1500, "-"), (1, 900, "+"), (1000, 1400, ".")],
             hits=[(900, 1, "s__A", 0.97, 1.04, "-"), (1500, 2500, "s__A", 0.91, 0.99, "+"),
                   (1000, 1400, "s__zz_unlisted", 0.99, 1.0, "+"), (850, 1450, "s__B", 0.85, 0.95, "+"),
                   (1, 2500, "Unknown", 0.7, 0.8, "+"), (10, 800, "s__A", 0.99, 0.5, "+")]),
        dict(loci=[(1, 600, "+"), (400, 1200, "-"), (1100, 1300, "+"), (1250, 1320, "+")],
             hits=[(1, 1200, "s__D", 0.9, 1.0, "+"), (380, 1310, "s__E", 0.88, 1.0, "-"),
                   (1100, 1320, "s__D", 0.7, 0.9, "+"), (1, 150, "s__F", 1.0, 1.0, "+")]),
        dict(loci=[(1, 500, "+")], hits=[]),
        dict(loci=[], hits=[(1, 500, "s__A", 0.9, 1.0, "+")]),
        dict(loci=[], hits=[]),
        dict(loci=[(1, 100, "+"), (150, 190, "-")], hits=[(1, 100, "s__A", 0.9, 1.0, "+")]),
        dict(loci=[(1, 1000, "+"), (1200, 2200, "+")],
             hits=[(1, 1000, "s__A", 0.45, 1.0, "+"), (1200, 2200, "s__A", 0.3, 1.0, "+")]),
        dict(loci=[(1, 1000, "+"), (1200, 2200, "+")],
             hits=[(1, 1000, "s__novel1", 0.95, 1.0, "+"), (1200, 2200, "s__novel2", 0.95, 1.0, "+")]),
        # scores the front end never produces but the ABI accepts: -0.0 and negative (the engine's integer
        # ranking of score bit patterns must fall back to floating-point compares for this contig)
        dict(loci=[(1, 1000, "+"), (1200, 2200, "+")],
             hits=[(1, 1000, "s__A", 0.9, 1.0, "+"), (1, 900, "s__A", -0.0, 1.0, "+"), (50, 1000, "s__A", -0.25, 1.0, "+"),
                   (1200, 2200, "s__A", 0.7, 1.0, "+"), (1200, 2100, "s__B", -0.0, 1.0, "+"),
                   (1250, 2200, "s__B", 0.0, 1.0, "+"), (1200, 2200, "s__D", 0.7, 1.0, "+")]),
    ]
    out["odd_inputs"] = make_batch(cs, TAX8)
    return out


ADVERSARIAL_FLAGS = [
    {}, dict(weak_loci="assign-unknown"), dict(weak_loci="penalize"),
    dict(one_clade_threshold=0.8, two_clade_threshold=0.5),
    dict(disambiguate_one="report-best", disambiguate_two="report-best", sister_penalty="off"),
    dict(disambiguate_two="jump", range=0.2, allow_lca=True),
    dict(stranded=True, min_overlap=0.5), dict(min_gene_length=0.0, min_scov=0.0, clade_genes=2),
    dict(jump_taxonomy=1, clade_leaves=2, ambiguous_threshold="off", sister_penalty="lenient"),
    dict(ambiguous_threshold="strict", annotation_threshold="strict", range=0.0),
]
