"""--write-details without a GPU: the details oracle against the golden tables of the reference's write_details, the
multi-member gzip layout of the details files, and the streamed CLIs accepting the flag."""
import gzip
import json
import os

import pytest

import helpers
from oracle import details_oracle
from waafle_b200 import streaming, writer

HEADER = "CONTIG_NAME\tITERATION\tCLADE\tGENE_SCORES\tGENE_SPANS\n"


def oracle_table(files, flags):
    """The details table (header included) the oracle derives for the demo inputs, contigs in blastout order."""
    from waafle_b200 import utils
    batch, loci, hits, tax = helpers.frontend_load(files)
    params = helpers.params_for(flags).as_dict()
    det = details_oracle.score_details(params, tax.tables(), batch.arrays())
    lengths = utils.read_contig_lengths(files["contigs"])
    order = streaming.details_order(batch, hits, lengths)
    return HEADER + details_oracle.details_text(det, batch.contig_names, tax.names, order)


@pytest.mark.parametrize("gff", ["genecaller", "prodigal"])
def test_oracle_details_equal_golden(tmp_path, gff):
    """The oracle's rows == the unmodified write_details (tests/golden/demo_cli/details_*.tsv.gz) for the 3 flag sets."""
    root = os.path.join(helpers.GOLDEN, "demo_cli")
    flag_sets = json.load(open(os.path.join(root, "details_flag_sets.json")))
    files = helpers.demo_files(tmp_path, gff == "prodigal")
    for k, flags in enumerate(flag_sets):
        with gzip.open(os.path.join(root, "details_{}_{}.tsv.gz".format(gff, k)), "rt") as fh:
            want = fh.read()
        got = oracle_table(files, flags)
        assert got == want, (gff, flags)
        assert got.count("\n") > 50


def test_multi_member_gzip_reads_back(tmp_path):
    """Header member + shards (one empty, one cut into several members) == the concatenated text."""
    text1 = "".join("c{}\t1\tk__A\t0.500|0.000\tNone|2:9\n".format(i) for i in range(5000)).encode()
    text2 = b"z\t2\tk__B\t1.000\t--\n"
    shards = []
    for k, pieces in enumerate([[text1[:7000], text1[7000:]], [], [text2]]):
        path = str(tmp_path / "s{}.gz".format(k))
        writer.write_details_file(path, iter(pieces), header=False)
        shards.append(path)
    assert os.path.getsize(shards[1]) == 0
    out = str(tmp_path / "all.tsv.gz")
    old = writer.DETAILS_BLOCK
    writer.DETAILS_BLOCK = 4096   # several members per piece
    try:
        writer.write_details_file(str(tmp_path / "one.tsv.gz"), iter([text1, b"", text2]))
    finally:
        writer.DETAILS_BLOCK = old
    writer.concat_details_shards(out, shards)
    want = HEADER + (text1 + text2).decode()
    for path in (out, str(tmp_path / "one.tsv.gz")):
        with gzip.open(path, "rt") as fh:
            assert fh.read() == want


@pytest.mark.parametrize("cli", ["orgscorer", "pipeline"])
def test_streamed_cli_accepts_write_details(cli):
    """--write-details with --devices / --stream-mb parses and is a streamed run (the flag no longer ends the run)."""
    from waafle_b200 import orgscorer, pipeline
    pos = ["c.fna", "b.blastout", "g.gff", "t.tsv"] if cli == "orgscorer" else ["c.fna", "b.blastout", "t.tsv"]
    mod = orgscorer if cli == "orgscorer" else pipeline
    for extra in (["--devices", "0,1"], ["--stream-mb", "4"]):
        args = mod.get_args(pos + ["--write-details"] + extra)
        assert args.write_details and orgscorer.streamed(args)
    assert not hasattr(orgscorer, "check_flags")
