"""GPU: the --write-details table built on the device (wfl_details.cu) against the details oracle, its "{:.3f}"
formatter against Python, bounded pieces, and streamed / multi-worker runs against the single call."""
import gzip
import os

import numpy as np
import pytest

import helpers
from oracle import details_oracle
from waafle_b200 import synth
from waafle_b200.engine import Engine, EngineError

pytestmark = pytest.mark.gpu

FLAG_SETS = [{}, {"weak_loci": "assign-unknown"}, {"weak_loci": "penalize"}, {"jump_taxonomy": 1},
             {"jump_taxonomy": 2, "weak_loci": "assign-unknown"}, {"stranded": True}, {"min_overlap": 0.0},
             {"min_gene_length": 1500.0}]


def device_text(batch, tax, params, order, wire="wide", piece_bytes=256 << 20, options=()):
    eng = Engine(0, params, tax)
    try:
        for k, v in options:
            eng.set_option(k, v)
        arrays = batch.to_packed(params.min_scov) if wire == "packed" else batch
        eng.score_batch_details(arrays, download=False)
        text = b"".join(eng.details_text(order, batch.contig_names, piece_bytes)).decode()
        return text, eng.stats(), eng.details_times
    finally:
        eng.close()


def oracle_text(batch, tax, params, order):
    det = details_oracle.score_details(params.as_dict(), tax.tables(), batch.arrays())
    return details_oracle.details_text(det, batch.contig_names, tax.names, order)


def check_equal(got, want, what):
    if got != want:
        g, w = got.split("\n"), want.split("\n")
        bad = next((i for i in range(min(len(g), len(w))) if g[i] != w[i]), min(len(g), len(w)) - 1)
        raise AssertionError((what, len(g), len(w), g[bad][:300], w[bad][:300]))


def synthetic(cfg, n, seed):
    data = synth.generate_config(cfg, n_contigs=n, seed=seed, **({"annotations": True} if cfg == "cfg5" else {}))
    tax = data.taxonomy()
    return data.to_batch(tax), tax, 1 if cfg == "cfg5" else 0


@pytest.mark.parametrize("cfg,n", [("cfg2", 100), ("cfg3", 30), ("cfg5", 30)])
def test_device_details_equal_oracle_on_synthetic(cfg, n):
    """Every flag set, both wire formats where the batch packs; rows in a shuffled contig order that leaves contigs out."""
    batch, tax, S = synthetic(cfg, n, 11)
    rng = np.random.default_rng(5)
    order = [int(c) for c in rng.permutation(batch.n_contigs)[: batch.n_contigs - 3]]
    wires = ["wide"] + (["packed"] if batch.can_pack(len(tax.names), S) else [])
    assert len(wires) == 2
    for flags in FLAG_SETS:
        params = helpers.params_for(flags, S)
        want = oracle_text(batch, tax, params, order)
        assert want.count("\n") > n
        for wire in wires:
            got, st, _ = device_text(batch, tax, params, order, wire)
            check_equal(got, want, (cfg, flags, wire))


def hand_built():
    """Contigs for the span rules (see the comments), the edge cases of which contigs have rows, and their taxonomy."""
    L = [(1001, 2000, "+"), (2101, 3000, "+")]
    contigs = [
        # single locus: one clade whose only hit scores 0 (empty cell -> `--`), one with a real run
        dict(loci=[(1, 1000, "+")], hits=[(1, 900, "s__A", 0.9, 0.9, "+"), (1, 900, "s__C", 0.0, 0.9, "+")]),
        # touching slices [0, 100) + [100, 200) merge; overlapping ones too; a one-site run is dropped; score <= 0
        dict(loci=L, hits=[(1001, 1100, "s__A", 0.9, 0.9, "+"), (1101, 1200, "s__A", 0.8, 0.9, "+"),
                           (1150, 1400, "s__A", 0.7, 0.9, "+"), (1700, 1700, "s__A", 0.9, 0.9, "+"),
                           (2101, 2900, "s__B", 0.9, 0.9, "+"), (2101, 2900, "s__D", -0.2, 0.9, "+"),
                           (1001, 1999, "s__D", 0.0, 0.9, "+"), (2101, 2600, "t__A1", 0.9, 0.9, "-")]),
        # a hit ending 200 sites before its locus: attaches under --min-overlap 0, and its python slice [0 : -200] wraps to
        # the locus's first 800 sites
        dict(loci=[(5001, 6000, "+"), (7001, 8000, "+")],
             hits=[(4500, 4800, "s__G", 0.9, 0.9, "+"), (5001, 5990, "s__E", 0.95, 0.9, "+"),
                   (7001, 7990, "s__F", 0.95, 0.9, "+"), (7001, 7500, "s__G", 0.6, 0.9, "+")]),
        # every locus weak: ignored under --weak-loci ignore (no rows), evaluated otherwise
        dict(loci=L, hits=[(1001, 1300, "s__A", 0.2, 0.9, "+"), (2101, 2300, "s__B", 0.2, 0.9, "+")]),
        # in the FASTA, without hits: never evaluated
        dict(loci=L, hits=[]),
        # two clades of one genus that need lifts
        dict(loci=L, hits=[(1001, 2000, "s__A", 0.9, 0.9, "+"), (1001, 2000, "s__B", 0.9, 0.9, "+"),
                           (2101, 3000, "s__D", 0.9, 0.9, "+"), (2101, 3000, "s__E", 0.9, 0.9, "+")]),
    ]
    return helpers.make_batch(contigs, helpers.TAX8)


@pytest.mark.parametrize("wire", ["wide", "packed"])
def test_device_details_equal_oracle_on_hand_built(wire):
    batch, tax = hand_built()
    order = list(range(batch.n_contigs))[::-1]
    seen = set()
    for flags in FLAG_SETS + [{"min_overlap": 0.0, "weak_loci": "assign-unknown"}]:
        params = helpers.params_for(flags)
        want = oracle_text(batch, tax, params, order)
        got, _, _ = device_text(batch, tax, params, order, wire)
        check_equal(got, want, (flags, wire))
        seen.add(want)
        names = {ln.split("\t")[0] for ln in got.splitlines()}
        assert "c00004" not in names   # no hits
        if not flags:
            assert "c00003" not in names   # every locus ignored
            rows = got.splitlines()
            assert any(r.startswith("c00000\t1\ts__C\t0.000\t--") for r in rows)
            assert any(r.startswith("c00001\t1\ts__A\t") and r.endswith("\t1:400|None") for r in rows)
        if flags == {"min_overlap": 0.0}:
            assert any(r.startswith("c00002\t1\ts__G\t") and r.endswith("\t1:800|1:500") for r in got.splitlines())
    assert len(seen) == len(FLAG_SETS) + 1


def test_replayed_contigs_give_one_copy_of_their_rows():
    """A tiny K2 group list makes the exact pipeline replay contigs; the dump then holds levels twice."""
    batch, tax, S = synthetic("cfg3", 30, 3)
    params = helpers.params_for({"weak_loci": "assign-unknown"}, S)
    order = list(range(batch.n_contigs))
    want = oracle_text(batch, tax, params, order)
    got, st, _ = device_text(batch, tax, params, order, options=[("k2_cap", 64)])
    assert st["workspace_retries"] > 0
    check_equal(got, want, "replay")


def test_bounded_pieces_give_the_same_text():
    batch, tax, S = synthetic("cfg2", 60, 4)
    params = helpers.params_for({"jump_taxonomy": 1}, S)
    order = list(range(batch.n_contigs))
    whole, _, t1 = device_text(batch, tax, params, order)
    tiny, _, t2 = device_text(batch, tax, params, order, piece_bytes=1)
    assert tiny == whole and t1["pieces"] == 1 and t2["pieces"] == len({ln.split("\t")[0] for ln in whole.splitlines()})


def test_formatter_equals_python():
    eng = Engine(0)
    try:
        rng = np.random.default_rng(7)
        ties = [k / 16.0 for k in range(1, 33, 2)]
        edges = []
        for k in range(2000):
            b = (k + 0.5) / 1000.0
            edges += [b, float(np.nextafter(b, 0.0)), float(np.nextafter(b, 3.0))]
        special = [0.0, -0.0, 1.0, -1.0, 5e-324, -5e-324, 2.2250738585072014e-308, -1e-300, -0.0004, -0.0005,
                   -0.0006, 0.9995, 1.9995, 2.0 ** 53 - 1, -(2.0 ** 53 - 1), 123456.7895]
        xs = np.array(ties + edges + special + list(rng.uniform(-2.0, 2.0, 1_000_000)), np.float64)
        got = eng.debug_format_scores(xs)
        want = ["{:.3f}".format(float(x)) for x in xs]
        bad = [i for i in range(len(xs)) if got[i] != want[i]]
        assert not bad, [(repr(float(xs[i])), got[i], want[i]) for i in bad[:5]]
        assert got[:3] == ["0.062", "0.188", "0.312"] and got[len(ties) + len(edges) + 1] == "-0.000"
        for x in (2.0 ** 53, -(2.0 ** 53), float("inf"), float("nan")):
            with pytest.raises(EngineError, match=r"error -6"):
                eng.debug_format_scores(np.array([1.0, x]))
    finally:
        eng.close()


def test_details_state_errors():
    batch, tax = hand_built()
    eng = Engine(0, helpers.params_for({}), tax)
    try:
        with pytest.raises(EngineError, match=r"error -3"):
            list(eng.details_text([0], batch.contig_names))
        eng.score_batch(batch)
        with pytest.raises(EngineError, match=r"error -3"):
            list(eng.details_text([0], batch.contig_names))
    finally:
        eng.close()


def read_details(outdir, basename):
    with gzip.open(os.path.join(str(outdir), basename + ".details.tsv.gz"), "rt") as fh:
        return fh.read()


@pytest.mark.parametrize("cli", ["orgscorer", "pipeline"])
def test_streamed_details_equal_single_call(tmp_path, cli):
    """--write-details with --stream-mb small and two workers == the single call; a FASTA-only contig has no rows."""
    from waafle_b200 import orgscorer, pipeline
    data = synth.generate_config("cfg5", n_contigs=150, seed=21, annotations=True)
    files = data.write_files(str(tmp_path), "s")
    with open(files["contigs"], "a") as fh:
        fh.write(">zz_fasta_only\nACGTACGTAC\n")
    pos = [files["contigs"], files["blastout"]] + ([files["gff"]] if cli == "orgscorer" else []) + [files["taxonomy"]]
    main = orgscorer.main if cli == "orgscorer" else pipeline.main
    mb = "{:.3f}".format(os.path.getsize(files["blastout"]) / 7.0 / (1 << 20))
    out = {}
    for tag, extra in (("one", []), ("streamed", ["--stream-mb", mb, "--devices", "0,0"])):
        outdir = tmp_path / tag
        outdir.mkdir()
        main(pos + ["--outdir", str(outdir), "--basename", "run", "--quiet", "--write-details",
                    "--weak-loci", "assign-unknown"] + extra)
        out[tag] = read_details(outdir, "run")
    assert out["one"] == out["streamed"]
    assert out["one"].count("\n") > 1000 and "zz_fasta_only" not in out["one"]
    assert out["one"].startswith("CONTIG_NAME\tITERATION\tCLADE\tGENE_SCORES\tGENE_SPANS\n")
