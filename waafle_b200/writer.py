"""Result unpacking and the three main TSV outputs.

Turns the engine's compacted result arrays back into the rows the reference writes in
`write_main_output_files` (waafle/waafle_orgscorer.py:814-894): same columns, same field
encodings (OS:750-764, 793-800), same float formatting and `--` for empty cells
(waafle/utils.py:137-139), rows sorted by contig name (OS:838).
"""

import collections
import concurrent.futures
import os
import shutil
import zlib

import numpy as np

from .utils import format_field, say, write_row

CALLS = ("unclassified", "no_lgt", "lgt")
FLAG_RETAINED, FLAG_IGNORED = 1, 2

C_ANNOTATION_PREFIX = "ANNOTATIONS:"   # OS:60
C_MISSING_ANNOTATION = "None"          # OS:61
DIRECTIONS = ("A?B", "B>A")            # OS:485, OS:543

# OS:78-114
FORMATS = {
    "lgt": ["contig_name", "call", "contig_length", "min_max_score", "avg_max_score", "synteny",
            "direction", "clade_A", "clade_B", "lca", "melded_A", "melded_B", "taxonomy_A",
            "taxonomy_B", "loci"],
    "no_lgt": ["contig_name", "call", "contig_length", "min_score", "avg_score", "synteny",
               "clade", "melded", "taxonomy", "loci"],
    "unclassified": ["contig_name", "call", "contig_length", "loci"],
}


def _tails_field(taxonomy, members, lca):
    """OS:750-759 on the distinct melded clades."""
    items = set()
    for m in members:
        t = taxonomy.get_tail(int(m), int(lca))
        if len(t) > 0:
            items.add("|".join(t))
    return "; ".join(sorted(items))


def _winner_annotations(batch, hits, res, systems):
    """{(locus row j, system index s): value} for every transferred annotation.  The subject headers of all
    winning hits are fetched and parsed once (they live in an Arrow array on the fast front end)."""
    aw = np.asarray(res["ann_winner"])
    if aw.ndim != 2 or aw.shape[1] == 0 or hits is None or not systems:
        return {}
    jj, ss = np.nonzero(aw >= 0)
    if len(jj) == 0:
        return {}
    rows = np.asarray(batch.hit_row)[aw[jj, ss]]
    sid = rows if hits.sseqid_id is None else np.asarray(hits.sseqid_id)[rows]   # None: one header per row (GPU parser)
    uniq = np.unique(sid)
    parsed = {int(u): hits.sseqid_annotations[int(u)] for u in uniq}
    return {(int(j), int(s)): parsed[int(i)][systems[int(s)]] for j, s, i in zip(jj.tolist(), ss.tolist(), sid.tolist())}


def build_records(batch, loci, hits, taxonomy, res):
    """One dict per contig (FASTA order) with the reference's row values, unformatted."""
    names = taxonomy.names
    S = res["ann_winner"].shape[1] if res["ann_winner"].ndim == 2 else 0
    systems = list(hits.systems)[:S] if hits is not None else []
    # plain Python lists: the loop below touches every element once, and numpy scalar access is ~10x slower
    locus_off = np.asarray(batch.locus_off).tolist()
    flags = np.asarray(res["locus_flags"]).tolist()
    locus_row = np.asarray(batch.locus_row).tolist()
    calls = np.asarray(res["call"]).tolist()
    lifts = np.asarray(res["lifts"]).tolist()
    lengths = np.asarray(batch.contig_lengths).tolist()
    member_off = np.asarray(res["member_off"]).tolist()
    n_members_a = np.asarray(res["n_members_a"]).tolist()
    members = np.asarray(res["members"]).tolist()
    clade1, clade2, lca = (np.asarray(res[k]).tolist() for k in ("clade1", "clade2", "lca"))
    crit, rank = np.asarray(res["crit"]).tolist(), np.asarray(res["rank"]).tolist()
    direction = np.asarray(res["direction"]).tolist()
    synteny = bytes(np.asarray(res["synteny"], dtype=np.uint8)).decode("latin-1")
    winners = _winner_annotations(batch, hits, res, systems)
    lineage_cache = {}

    def lineage(c):
        if c not in lineage_cache:
            lineage_cache[c] = "|".join(taxonomy.get_lineage(c))
        return lineage_cache[c]

    records = []
    for c in range(batch.n_contigs):
        l0, l1 = locus_off[c], locus_off[c + 1]
        kept = [j for j in range(l0, l1) if flags[j] & FLAG_RETAINED]
        rec = dict(
            contig_name=batch.contig_names[c], call=CALLS[calls[c]],
            contig_length=lengths[c],
            loci="|".join(loci.code(locus_row[j]) for j in kept),
            ignore=[bool(flags[j] & FLAG_IGNORED) for j in kept],
            lifts=lifts[c])
        ann = []
        for j in kept:
            d = {}
            for s in range(S):
                v = winners.get((j, s))
                if v is not None:
                    d[systems[s]] = v
            ann.append(d)
        rec["annotations"] = ann
        call = calls[c]
        if call:
            m0, m1 = member_off[c], member_off[c + 1]
            na = n_members_a[c]
            mem = members[m0:m1]
            c1 = clade1[c]
            syn = "".join(synteny[j] for j in kept)
            if call == 1:
                rec.update(min_score=crit[c], avg_score=rank[c],
                           synteny=syn, clade=names[c1],
                           melded=_tails_field(taxonomy, mem[:na], c1),
                           taxonomy=lineage(c1))
            else:
                c2 = clade2[c]
                rec.update(min_max_score=crit[c],
                           avg_max_score=rank[c], synteny=syn,
                           direction=DIRECTIONS[direction[c]],
                           clade_A=names[c1], clade_B=names[c2], lca=names[lca[c]],
                           melded_A=_tails_field(taxonomy, mem[:na], c1),
                           melded_B=_tails_field(taxonomy, mem[na:], c2),
                           taxonomy_A=lineage(c1),
                           taxonomy_B=lineage(c2))
        records.append(rec)
    return records


def write_main_output_files(records, outdir, basename):
    """Write <basename>.{lgt,no_lgt,unclassified}.tsv (OS:814-894)."""
    say("Initializing outputs.")
    # annotation systems that were actually transferred to some locus (OS:824-828)
    systems = sorted({s for r in records for d in r["annotations"] for s in d})
    handles = {}
    for option in ("lgt", "no_lgt", "unclassified"):
        handles[option] = open(os.path.join(outdir, ".".join([basename, option, "tsv"])), "w")
        cols = FORMATS[option] + [C_ANNOTATION_PREFIX + s for s in systems]
        write_row([k.upper() for k in cols], handles[option])
    for r in sorted(records, key=lambda r: r["contig_name"]):
        option = r["call"]
        cells = [format_field(r[f]) for f in FORMATS[option]]
        for s in systems:
            cells.append(format_field("|".join(d.get(s, C_MISSING_ANNOTATION)
                                               for d in r["annotations"])))
        write_row(cells, handles[option])
    for h in handles.values():
        h.close()


# ---------------------------------------------------------------------------------------------------------------
# --write-details (OS:766-812)
# ---------------------------------------------------------------------------------------------------------------

DETAILS_FORMAT = ["contig_name", "iteration", "clade", "gene_scores", "gene_spans"]   # OS:116-122
DETAILS_LEVEL = 6             # zlib's default level: about twice as fast as gzip's 9 for a few % more bytes
DETAILS_BLOCK = 16 << 20      # text per gzip member: the unit of parallel compression


def gzip_member(data, level=DETAILS_LEVEL):
    """`data` as one complete gzip member."""
    z = zlib.compressobj(level, zlib.DEFLATED, 31)
    return z.compress(data) + z.flush()


def write_gzip_members(fh, pieces, threads=None):
    """Concatenated gzip members of the byte strings `pieces` (cut into DETAILS_BLOCK blocks), compressed in a thread pool
    (zlib releases the GIL) while the next pieces are produced, written to the binary handle `fh` in order.  A
    multi-member file reads back with gzip.open like any gzip file."""
    threads = threads or min(32, os.cpu_count() or 1)
    pending = collections.deque()
    with concurrent.futures.ThreadPoolExecutor(threads) as pool:
        for piece in pieces:
            view = memoryview(piece)
            for i in range(0, len(view), DETAILS_BLOCK):
                pending.append(pool.submit(gzip_member, view[i:i + DETAILS_BLOCK]))
            while len(pending) > 2 * threads:
                fh.write(pending.popleft().result())
        while pending:
            fh.write(pending.popleft().result())
    return threads


def details_header():
    return ("\t".join(k.upper() for k in DETAILS_FORMAT) + "\n").encode()


def write_details_file(path, pieces, header=True):
    """<basename>.details.tsv.gz (OS:931-937, 802-812): the header row, then the rows the engine built on the device
    (Engine.details_text), as concatenated gzip members.  header=False writes a shard of a streamed run."""
    with open(path, "wb") as fh:
        if header:
            fh.write(gzip_member(details_header()))
        return write_gzip_members(fh, pieces)


def concat_details_shards(path, shards):
    """The header member, then the details shards of a streamed run in chunk (= blastout) order."""
    with open(path, "wb") as dst:
        dst.write(gzip_member(details_header()))
        for shard in shards:
            with open(shard, "rb") as src:
                shutil.copyfileobj(src, dst)
