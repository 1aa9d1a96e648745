"""
TEST INFRASTRUCTURE ONLY -- CPU oracle of the --write-details table (write_details, waafle_orgscorer.py:766-812).

It walks every contig through the classes of orgscorer_oracle (attach_hits, update_gene_scores, the --jump-taxonomy
lifts and the evaluate_contig loop, OS:566-583 / 952-960) and, at every evaluated level, takes the clade rows straight
from the contig's own gene scores and site arrays.  Nothing here reads the engine.
"""

import numpy as np

from oracle import orgscorer_oracle as O


def _details_rows(C, ev):
    """write_details (OS:802-812) at evaluation index `ev`: (ITERATION, clade, GENE_SCORES, GENE_SPANS) per clade in
    ascending node order.  ITERATION = max(1, ev) (OS:566-579); a span cell is None without a site array (OS:776-781),
    else the 1-based first and last site of every non-zero run of at least two sites (OS:773-791); an empty field
    prints `--` (UT:137-139)."""
    rows = []
    for clade in sorted(C.gene_scores):
        ld = C.site_scores.get(clade, {})
        cells = []
        for i in range(C.G):
            if i not in ld:
                cells.append("None")
                continue
            nz = np.r_[False, ld[i] != 0, False].astype(np.int8)
            edges = np.flatnonzero(np.diff(nz))
            cells.append(":".join("{}:{}".format(a + 1, b) for a, b in zip(edges[::2], edges[1::2]) if b - a >= 2))
        scores = "|".join("{:.3f}".format(v) for v in C.gene_scores[clade])
        spans = "|".join(cells)
        rows.append((max(1, ev), clade, scores or "--", spans or "--"))
    return rows


def score_details(params, tax, batch):
    """Per contig of the batch (same inputs as orgscorer_oracle.score_batch), its details rows in evaluation order."""
    P = dict(params)
    T = O._Tax(tax)
    n = len(batch["hit_off"]) - 1
    S = P["n_systems"]
    hsys = batch.get("hit_sysmask")
    out = []
    for c in range(n):
        h0, h1 = int(batch["hit_off"][c]), int(batch["hit_off"][c + 1])
        l0, l1 = int(batch["locus_off"][c]), int(batch["locus_off"][c + 1])
        C = O._Contig(P, T, batch["locus_start"][l0:l1], batch["locus_end"][l0:l1], batch["locus_strand"][l0:l1])
        rows = []
        if h1 > h0:   # contigs absent from the blastout are never visited (OS:943-960)
            C.attach_hits(batch["hit_qstart"][h0:h1], batch["hit_qend"][h0:h1], batch["hit_taxon"][h0:h1],
                          batch["hit_score"][h0:h1], batch["hit_scov"][h0:h1], batch["hit_strand"][h0:h1],
                          hsys[h0:h1] if (hsys is not None and S > 0) else None, h0)
            C.update_gene_scores()
            for _ in range(P["jump_taxonomy"]):   # OS:955-957
                C.raise_taxonomy()
            if not all(C.ignore):   # OS:959
                rows += _details_rows(C, 0)
                best_one = O._explain_one(C)
                best_two = O._explain_two(C) if not O._is_ok(best_one) else None
                it = 1
                while (len(C.clades) > 0 and T.root not in C.clades
                       and not O._is_ok(best_one) and not O._is_ok(best_two)):
                    C.raise_taxonomy()
                    rows += _details_rows(C, it)
                    best_one = O._explain_one(C)
                    best_two = O._explain_two(C) if not O._is_ok(best_one) else None
                    it += 1
                    if it > 100:
                        raise RuntimeError("Runaway taxonomic recursion")
        out.append(rows)
    return out


def details_text(details, contig_names, clade_names, order):
    """The rows of score_details as the table's text (no header): contigs in `order`."""
    out = []
    for c in order:
        for it, clade, scores, spans in details[c]:
            out.append("\t".join([contig_names[c], str(it), clade_names[clade], scores, spans]) + "\n")
    return "".join(out)
