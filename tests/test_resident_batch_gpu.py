"""GPU: the scoring batch built on the device from the parser's resident hit columns (wfl_upload_parsed,
csrc/wfl_resident_batch.cu) equals `packing.pack` byte for byte and scores the same; the CLIs take that path on
GPU-parsed blastouts and write the bytes of their --cpu-parse runs; bad inputs fail with their status and leave no
batch."""
import gzip
import os

import numpy as np
import pytest

import helpers
from test_compressed import bgzf
from waafle_b200 import compressed, engine, gpu_parse, packing, parsers, synth, taxonomy, utils
from waafle_b200.params import OrgscorerParams

pytestmark = pytest.mark.gpu
ROUTE = ("fallback_contigs", "second_pass_contigs", "smem_contigs", "fallback_reasons", "guard_trips", "refined_groups",
         "contigs", "hits", "loci")
WFL_ERR_ARG, WFL_ERR_STATE = -1, -3


@pytest.fixture(scope="module")
def parser():
    p = gpu_parse.BlastParser(0)
    yield p
    p.close()


def _tax(files, hits):
    return taxonomy.Taxonomy(files["taxonomy"]).build(hits.distinct_taxa())


def check_equal(hits, lengths, loci, tax, capfd=None, score=True):
    """Both batches of one parse: columns byte for byte, offsets and locus rows, and the results in both modes."""
    if capfd is not None:
        capfd.readouterr()
    host = packing.pack(lengths, loci, hits, tax)
    host_err = capfd.readouterr().err if capfd is not None else None
    res = packing.pack_resident(lengths, loci, hits, tax)
    if capfd is not None:
        assert capfd.readouterr().err == host_err   # the same "Unknown contig" lines
    for k in ("hit_off", "locus_off", "locus_row", "locus_start", "locus_end", "locus_strand", "contig_lengths"):
        assert np.array_equal(getattr(host, k), getattr(res, k)), k
    S = len(hits.systems)
    eng = engine.Engine(0, OrgscorerParams(n_systems=S), tax)
    eng.upload_parsed(res)
    got = eng.debug_resident_batch()
    want = host.arrays()
    assert sorted(got) == sorted(k for k in want if k.startswith("hit_") and k != "hit_off")
    for k, v in got.items():
        assert v.dtype == want[k].dtype and v.tobytes() == want[k].tobytes(), k
    if score:
        for mode in (0, 1):
            eng.set_option("exact", mode)
            a = eng.score_batch(host)
            sa = eng.stats()
            b = eng.score_batch(res)
            sb = eng.stats()
            assert sorted(a) == sorted(b)
            for k in a:
                assert np.array_equal(a[k], b[k]), (mode, k)
            for k in ROUTE:
                assert sa[k] == sb[k], (mode, k)
    eng.close()
    return host, res


@pytest.mark.parametrize("shape", ["cfg2", "cfg3", "cfg5"])
@pytest.mark.parametrize("annotations", [False, True])
def test_synthetic_shapes(tmp_path, parser, shape, annotations):
    data = synth.generate_config(shape, n_contigs=400, seed=61, annotations=annotations)
    files = data.write_files(str(tmp_path), shape)
    hits = parser.parse(open(files["blastout"], "rb").read())
    assert (hits.systems != []) == annotations
    check_equal(hits, utils.read_contig_lengths(files["contigs"]), parsers.read_gff_loci(files["gff"]), _tax(files, hits))


def test_fasta_order_unknown_and_hitless_contigs(tmp_path, parser, capfd):
    data = synth.generate_config("cfg2", n_contigs=300, seed=5, annotations=False)
    files = data.write_files(str(tmp_path), "o")
    lengths = utils.read_contig_lengths(files["contigs"])
    names = list(lengths)
    rng = np.random.default_rng(9)
    keep = [names[i] for i in rng.permutation(len(names))[:-11]]
    shuffled = {nm: lengths[nm] for nm in keep}
    shuffled.update({"no_hits_{}".format(k): 900 + k for k in range(5)})
    hits = parser.parse(open(files["blastout"], "rb").read())
    host, _ = check_equal(hits, shuffled, parsers.read_gff_loci(files["gff"]), _tax(files, hits), capfd)
    assert host.n_hits < len(hits) and (np.diff(host.hit_off) == 0).any()


def test_empty_blastout(tmp_path, parser):
    files = helpers.demo_files(tmp_path)
    hits = parser.parse(b"")
    assert len(hits) == 0 and gpu_parse.live_resident(hits) is not None
    host, res = check_equal(hits, utils.read_contig_lengths(files["contigs"]), parsers.read_gff_loci(files["gff"]),
                            _tax(files, hits))
    assert res.n_hits == 0 and res.n_loci > 0


def _rows(contig, n, rng, pident=None, taxa=8, reverse_every=0, qlen=200000):
    out = []
    for i in range(n):
        q1 = int(rng.integers(1, 60000))
        q2 = q1 + int(rng.integers(50, 3000))
        s1, s2 = 1, q2 - q1 + 1
        if reverse_every and i % reverse_every == 0:
            s1, s2 = s2, s1   # plus strand with send < sstart: scov < 0
        p = pident if pident is not None else "{:.3f}".format(rng.uniform(30, 100))
        out.append("\t".join(str(x) for x in (contig, "G{}|s__t{}".format(i, int(rng.integers(taxa))), qlen, s2 + s1, q2 - q1 + 1,
                                               q1, q2, s1, s2, p, 10, 0, "0.0", 100, "plus")))
    return out


def _case(rows, tmp_path, n_loci=3):
    """Blastout text of `rows` (a list of row lists, one per contig), its contig lengths, loci and taxonomy."""
    text = ("\n".join(r for block in rows for r in block) + "\n").encode()
    names = list(dict.fromkeys(r.split("\t", 1)[0] for block in rows for r in block))
    lengths = {nm: 200000 for nm in names}
    seq = [nm for nm in names for _ in range(n_loci)]
    loci = parsers.LocusTable(seq, [1 + 20000 * (k % n_loci) for k in range(len(seq))],
                              [15000 + 20000 * (k % n_loci) for k in range(len(seq))], ["+"] * len(seq))
    tax_path = os.path.join(str(tmp_path), "tax.tsv")
    with open(tax_path, "w") as fh:
        fh.write("".join("s__t{}\tg__g{}\n".format(k, k % 3) for k in range(64)))
        fh.write("".join("g__g{}\tr__Root\n".format(k) for k in range(3)))
    return text, lengths, loci, dict(taxonomy=tax_path)


def test_ties_zero_and_negative_scores(tmp_path, parser):
    rng = np.random.default_rng(4)
    cases = {
        # equal scores within a taxon: the same row repeated keeps file order
        "ties": [[_rows("c1", 1, rng, taxa=1)[0]] * 40 + _rows("c1", 30, rng, taxa=2), _rows("c2", 50, rng, "77.000", 3)],
        # every pident 0.000: smax = 0, the lexsort branch; scov < 0 gives -0.0 among the +0.0
        "zeros": [_rows("c{}".format(k), 60, rng, "0.000", 4, reverse_every=3) for k in range(6)],
        # negative scores among positive ones: clipped to 0 in the quantised key
        "negative": [_rows("c{}".format(k), 60, rng, None, 4, reverse_every=4) for k in range(6)],
    }
    for name, rows in cases.items():
        text, lengths, loci, files = _case(rows, tmp_path)
        hits = parser.parse(text)
        if name == "zeros":
            assert (np.signbit(hits.score) & (hits.score == 0)).any() and hits.score.max() == 0.0
        if name == "negative":
            assert (hits.score < 0).any() and hits.score.max() > 0
        check_equal(hits, lengths, loci, _tax(files, hits))


def test_contigs_beyond_the_first_launch(tmp_path, parser):
    """65 535- and 70 000-hit contigs among ordinary ones: their keys are sorted by the second launch."""
    rng = np.random.default_rng(8)
    rows = [_rows("a{}".format(k), int(rng.integers(1, 300)), rng) for k in range(40)]
    rows.insert(7, _rows("big1", 65535, rng, taxa=50))
    rows.insert(21, _rows("big2", 70000, rng, taxa=50))
    rows.append(_rows("c2047", 2047, rng))
    rows.append(_rows("c2049", 2049, rng))
    text, lengths, loci, files = _case(rows, tmp_path)
    hits = parser.parse(text)
    check_equal(hits, lengths, loci, _tax(files, hits))


def test_bgzf_sub_range(tmp_path, parser):
    data = synth.generate_config("cfg2", n_contigs=200, seed=12, annotations=False)
    files = data.write_files(str(tmp_path), "z")
    text = open(files["blastout"], "rb").read()
    raw = bgzf(text, block=9000)
    members = compressed.bgzf_members(raw)
    # a range of whole contig blocks from the middle of the text
    rows = text.split(b"\n")[:-1]
    row_off = np.r_[0, np.cumsum([len(r) + 1 for r in rows])]
    names = [r.split(b"\t", 1)[0] for r in rows]
    starts = [int(row_off[k]) for k in range(len(rows)) if k == 0 or names[k] != names[k - 1]]
    off, end = starts[len(starts) // 4], starts[3 * len(starts) // 4]
    hits = parser.parse_bgzf(raw, members, own=(off, end - off))
    assert hits is not None and 0 < len(hits) < text.count(b"\n")
    check_equal(hits, utils.read_contig_lengths(files["contigs"]), parsers.read_gff_loci(files["gff"]), _tax(files, hits))


def test_gene_call_and_gff_loci(tmp_path, parser):
    data = synth.generate_config("cfg5", n_contigs=200, seed=30, annotations=True)
    files = data.write_files(str(tmp_path), "g")
    hits = parser.parse(open(files["blastout"], "rb").read())
    gene_off, start, end, strand = parser.call_genes(0.1, 200, 0.75)
    calls = parsers.LocusTable.from_blocks(list(hits.block_names), gene_off, start, end, strand)
    lengths = utils.read_contig_lengths(files["contigs"])
    check_equal(hits, lengths, calls, _tax(files, hits))
    check_equal(hits, lengths, parsers.read_gff_loci(files["gff"], device=0), _tax(files, hits))


# ---- errors --------------------------------------------------------------------------------------------------------

def _demo(tmp_path, parser):
    files = helpers.demo_files(tmp_path)
    hits = parser.parse(open(files["blastout"], "rb").read())
    tax = _tax(files, hits)
    res = packing.pack_resident(utils.read_contig_lengths(files["contigs"]), parsers.read_gff_loci(files["gff"]), hits, tax)
    return files, hits, tax, res


def _fails(tax, res, status, S):
    eng = engine.Engine(0, OrgscorerParams(n_systems=S), tax)
    with pytest.raises(engine.EngineError, match="error {}:".format(status)):
        eng.upload_parsed(res)
    assert eng._lib.wfl_run_resident(eng._h) == WFL_ERR_STATE   # no batch left behind
    eng.close()


def test_errors_leave_no_batch(tmp_path, parser):
    files, hits, tax, res = _demo(tmp_path, parser)
    S = len(hits.systems)
    c = int(np.flatnonzero(np.diff(res.hit_off))[-1])
    bad = res.slice(0, res.n_contigs)
    bad.hit_src = res.hit_src.copy()
    bad.hit_src[c] = len(hits) - int(res.hit_off[c + 1] - res.hit_off[c]) + 1   # one row past the last
    _fails(tax, bad, WFL_ERR_ARG, S)
    for value in (-1, len(tax.names)):   # an unmapped slot, a node past the taxonomy
        bad = res.slice(0, res.n_contigs)
        bad.slot_node = res.slot_node.copy()
        bad.slot_node[res.resident.taxon_slots[0]] = value
        _fails(tax, bad, WFL_ERR_ARG, S)
    bad = res.slice(0, res.n_contigs)
    c = int(np.flatnonzero(np.diff(res.hit_off) > 1)[0])
    bad.hit_off = res.hit_off.copy()
    bad.hit_off[c + 1] = bad.hit_off[c + 2] + 1   # not monotone
    _fails(tax, bad, WFL_ERR_ARG, S)
    # the parser's last parse flagged a row: the batch's parse is gone, and a clean-looking generation does not help
    assert parser.parse(b'c1\t"quoted"\t1\t1\t1\t1\t1\t1\t1\t1\t1\t1\t1\t1\tplus\n') is None
    with pytest.raises(engine.EngineError, match="no longer live"):
        engine.Engine(0, OrgscorerParams(n_systems=S), tax).upload_parsed(res)
    res.resident.generation = parser.generation
    _fails(tax, res, WFL_ERR_STATE, S)


def test_stale_generation(tmp_path, parser):
    files, hits, tax, res = _demo(tmp_path, parser)
    parser.parse(open(files["blastout"], "rb").read())
    assert gpu_parse.live_resident(hits) is None
    eng = engine.Engine(0, OrgscorerParams(n_systems=len(hits.systems)), tax)
    with pytest.raises(engine.EngineError, match="no longer live"):
        eng.score_batch(res)
    assert eng._lib.wfl_run_resident(eng._h) == WFL_ERR_STATE
    eng.close()


def test_parser_on_another_device(tmp_path):
    if engine.load_library().wfl_device_count() < 2:
        pytest.skip("needs two GPUs")
    p1 = gpu_parse.BlastParser(1)
    files, hits, tax, res = _demo(tmp_path, p1)
    _fails(tax, res, WFL_ERR_ARG, len(hits.systems))
    p1.close()


# ---- the CLIs ------------------------------------------------------------------------------------------------------

def _outputs(outdir, details=False):
    got = {k: open(os.path.join(str(outdir), "run.{}.tsv".format(k))).read() for k in ("lgt", "no_lgt", "unclassified")}
    if details:
        with gzip.open(os.path.join(str(outdir), "run.details.tsv.gz"), "rt") as fh:
            got["details"] = fh.read()
    return got


@pytest.fixture
def count_pack(monkeypatch):
    calls = []
    real = packing.pack

    def pack(*a, **k):
        calls.append(1)
        return real(*a, **k)
    monkeypatch.setattr(packing, "pack", pack)
    return calls


def test_cli_single_calls_take_the_resident_path(tmp_path, count_pack, capfd):
    from waafle_b200 import orgscorer, pipeline
    data = synth.generate_config("cfg5", n_contigs=300, seed=44, annotations=True)
    files = data.write_files(str(tmp_path), "run")
    plain = synth.generate_config("cfg2", n_contigs=300, seed=45, annotations=False).write_files(str(tmp_path / "p"), "run")
    runs = [("org", files, []), ("org", plain, []), ("org", plain, ["--write-details"]),
            ("org", plain, ["--chunk-contigs", "37"]), ("org", files, ["--exact-scores", "--chunk-contigs", "50"]),
            ("pipe", plain, []), ("pipe", files, ["--write-details"])]
    for k, (cli, f, flags) in enumerate(runs):
        outs, errs = {}, {}
        for tag, extra in (("gpu", []), ("cpu", ["--cpu-parse"])):
            out = tmp_path / "o{}_{}".format(k, tag)
            out.mkdir()
            del count_pack[:]
            if cli == "org":
                orgscorer.main([f["contigs"], f["blastout"], f["gff"], f["taxonomy"], "--outdir", str(out),
                                "--basename", "run"] + flags + extra)
            else:
                pipeline.main([f["contigs"], f["blastout"], f["taxonomy"], "--outdir", str(out), "--basename", "run"]
                              + flags + extra)
            assert (len(count_pack) == 0) == (tag == "gpu"), (cli, flags, tag)
            outs[tag] = _outputs(out, "--write-details" in flags)
            errs[tag] = [ln for ln in capfd.readouterr().err.splitlines() if not ln.startswith("  ")]
        assert outs["gpu"] == outs["cpu"], (cli, flags)
        assert errs["gpu"] == errs["cpu"], (cli, flags)   # the stage lines


def test_cli_flagged_row_falls_back_to_the_host_pack(tmp_path, count_pack):
    from waafle_b200 import orgscorer
    files = helpers.demo_files(tmp_path)
    text = open(files["blastout"]).read().split("\n")
    f = text[3].split("\t")
    f[9] = "9.87e1"   # an exponent float: the device parser flags the row
    text[3] = "\t".join(f)
    path = str(tmp_path / "flagged.blastout")
    with open(path, "w") as fh:
        fh.write("\n".join(text))
    outs = {}
    for tag, extra in (("gpu", []), ("cpu", ["--cpu-parse"])):
        out = tmp_path / tag
        out.mkdir()
        del count_pack[:]
        orgscorer.main([files["contigs"], path, files["gff"], files["taxonomy"], "--outdir", str(out), "--basename", "run",
                        "--quiet"] + extra)
        assert len(count_pack) == 1
        outs[tag] = _outputs(out)
    assert outs["gpu"] == outs["cpu"]


def test_chunk_scorer_takes_the_resident_path(tmp_path, count_pack):
    """The streamed workers' scorer: a chunk parsed on its GPU is packed on the device, text and BGZF alike."""
    from waafle_b200 import orgscorer, streaming
    data = synth.generate_config("cfg5", n_contigs=200, seed=46, annotations=True)
    files = data.write_files(str(tmp_path), "run")
    args = orgscorer.get_args([files["contigs"], files["blastout"], files["gff"], files["taxonomy"]])
    tax = taxonomy.Taxonomy(files["taxonomy"])
    lengths = utils.read_contig_lengths(files["contigs"])
    index = streaming.LociIndex(parsers.read_gff_loci(files["gff"]), lengths)
    text = open(files["blastout"], "rb").read()
    raw = bgzf(text, block=9000)
    members = compressed.bgzf_members(raw)
    records = {}
    for tag in ("text", "bgzf", "cpu"):
        scorer = streaming.ChunkScorer(0, args, tax, lengths, index, functools_partial(args), cpu_parse=tag == "cpu")
        del count_pack[:]
        hits = scorer.parse_bgzf(raw, members, 0, len(text)) if tag == "bgzf" else scorer.parse(text)
        recs, names = scorer.score(streaming.chunk_contigs(hits, lengths), hits)
        assert (len(count_pack) == 0) == (tag != "cpu"), tag
        records[tag] = (recs, names)
        scorer.close()
    assert repr(records["text"]) == repr(records["cpu"]) == repr(records["bgzf"])


def functools_partial(args):
    import functools
    from waafle_b200 import orgscorer
    return functools.partial(orgscorer.params_from_args, args)


def test_streamed_runs_equal_cpu_parse(tmp_path):
    from waafle_b200 import orgscorer
    data = synth.generate_config("cfg2", n_contigs=300, seed=47, annotations=False)
    files = data.write_files(str(tmp_path), "run")
    gz = str(tmp_path / "run.blastout.gz")
    with open(files["blastout"], "rb") as fh, open(gz, "wb") as dst:
        dst.write(bgzf(fh.read(), block=7000))
    outs = []
    for blastout, extra in ((files["blastout"], []), (gz, []), (files["blastout"], ["--cpu-parse"])):
        out = tmp_path / "s{}".format(len(outs))
        out.mkdir()
        orgscorer.main([files["contigs"], blastout, files["gff"], files["taxonomy"], "--outdir", str(out), "--basename",
                        "run", "--quiet", "--stream-mb", "0.05", "--devices", "0,0", "--write-details"] + extra)
        outs.append(_outputs(out, True))
    assert outs[0] == outs[2] and outs[1] == outs[2]
