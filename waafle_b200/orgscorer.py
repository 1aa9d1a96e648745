"""`waafle_orgscorer` front end over the B200 engine.

Same positional arguments and flags as the reference CLI (waafle/waafle_orgscorer.py:135-303 plus
the shared flags of waafle/waafle_genecaller.py:81-101), same stderr stage messages, same three
output TSVs.  The only part that differs is the body of the major contig loop
(waafle_orgscorer.py:952-960), which is one `Engine.score_batch` call on the GPU.
`--write-details` writes <basename>.details.tsv.gz with the content the reference's write_details (OS:766-812) produces
when given a text-mode handle (upstream opens the gzip in binary mode and fails on Python 3).
"""

import argparse
import functools
import os
import sys

from . import gpu_parse, packing, parsers, taxonomy, writer
from .engine import Engine
from .params import OrgscorerParams
from .utils import die, read_contig_lengths, say


def get_args(argv=None):
    parser = argparse.ArgumentParser(
        description="Step 2 in the WAAFLE pipeline: merge blast hits into genes on contigs and "
                    "identify contigs best explained by one clade vs. a pair of clades (putative LGT). "
                    "B200-native engine.",
        formatter_class=argparse.RawTextHelpFormatter)
    g = parser.add_argument_group("required inputs")
    g.add_argument("contigs", help="contigs file (.fasta format)")
    g.add_argument("blastout", help="output of waafle_search for one set of contigs (.blastout)")
    g.add_argument("gff", help="gene calls (from waafle_genecaller or user-supplied) for <contigs> (.gff)")
    g.add_argument("taxonomy", help="taxonomy file for the blast database used to make <blastout>")
    add_flags(parser)
    return parser.parse_args(argv)


def add_flags(parser):
    """The orgscorer's optional flags (everything but the positional inputs), added to `parser`."""
    g = parser.add_argument_group("output formatting")
    g.add_argument("--outdir", default=".", metavar="<path>")
    g.add_argument("--basename", default=None, metavar="<str>")
    g.add_argument("--write-details", action="store_true")
    g.add_argument("--quiet", action="store_true")
    g = parser.add_argument_group("main parameters")
    g.add_argument("-k1", "--one-clade-threshold", type=float, default=0.5, metavar="<0.0-1.0>")
    g.add_argument("-k2", "--two-clade-threshold", type=float, default=0.8, metavar="<0.0-1.0>")
    g.add_argument("--disambiguate-one", choices=["report-best", "meld"], default="meld")
    g.add_argument("--disambiguate-two", choices=["report-best", "jump", "meld"], default="meld")
    g.add_argument("--range", type=float, default=0.05, metavar="<float>")
    g.add_argument("--jump-taxonomy", type=int, default=None, metavar="<1-N>")
    g = parser.add_argument_group("post-detection LGT filters")
    g.add_argument("--allow-lca", action="store_true")
    g.add_argument("--ambiguous-fraction", type=float, default=0.1, metavar="<0.0-1.0>")
    g.add_argument("--ambiguous-threshold", choices=["off", "lenient", "strict"], default="lenient")
    g.add_argument("--sister-penalty", choices=["off", "lenient", "strict"], default="strict")
    g.add_argument("--clade-genes", type=int, default=None, metavar="<1-N>")
    g.add_argument("--clade-leaves", type=int, default=None, metavar="<1-N>")
    g = parser.add_argument_group("gene-hit merge parameters")
    g.add_argument("--weak-loci", choices=["ignore", "penalize", "assign-unknown"], default="ignore")
    g.add_argument("--annotation-threshold", choices=["off", "lenient", "strict"], default="lenient")
    g.add_argument("--min-overlap", type=float, default=0.1, metavar="<0.0-1.0>")
    g.add_argument("--min-gene-length", default=200, type=float, metavar="<int>")
    g.add_argument("--min-scov", default=0.75, type=float, metavar="<float>")
    g.add_argument("--stranded", action="store_true")
    g = parser.add_argument_group("engine")
    g.add_argument("--device", type=int, default=0, help="CUDA device index [default: 0]")
    g.add_argument("--cpu-parse", action="store_true",
                   help="parse the blastout with the CPU reader instead of the CUDA parser")
    g.add_argument("--chunk-contigs", type=int, default=250000,
                   help="contigs per engine call (streaming; results are merged) [default: 250000]")
    g.add_argument("--exact-scores", action="store_true",
                   help="score every contig with the exact (numpy summation order) pipeline: min/avg scores bit-identical to\n"
                        "the reference instead of within 1e-12 [default: fused fast path with guard bands]")
    g.add_argument("--devices", default=None, metavar="<0,1,...|all>",
                   help="CUDA devices for a streamed run: the blastout is cut into contig-aligned chunks that are parsed,\n"
                        "scored and written by one worker process per device, then merged by contig name\n"
                        "[default: the single --device, whole file in one pass]")
    g.add_argument("--stream-mb", type=float, default=0.0, metavar="<MB>",
                   help="blastout text per streamed chunk; > 0 streams even on one device [default: 256 with --devices]")


def streamed(args):
    return args.devices is not None or args.stream_mb > 0


def params_from_args(args, n_systems):
    return OrgscorerParams.from_args(args, n_systems=n_systems)


def device_list(spec, default):
    """`--devices` -> list of CUDA device indices, without touching CUDA in this process (the workers are forks)."""
    if spec is None:
        return [default]
    if spec == "all":
        import subprocess
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout
        n = sum(1 for ln in out.splitlines() if ln.startswith("GPU "))
        if n == 0:
            die("--devices all: nvidia-smi lists no GPU")
        return list(range(n))
    try:
        return [int(x) for x in spec.split(",") if x != ""]
    except ValueError:
        die("bad --devices:", spec)


def score_in_chunks(engine, batch, chunk):
    """Contigs are independent, so a long run is scored chunk by chunk and concatenated."""
    import numpy as np
    if batch.n_contigs <= chunk:
        return engine.score_batch(batch)
    parts, c0 = [], 0
    while c0 < batch.n_contigs:
        c1 = min(batch.n_contigs, c0 + chunk)
        r = engine.score_batch(batch.slice(c0, c1))
        r["ann_winner"] = np.where(r["ann_winner"] >= 0, r["ann_winner"] + int(batch.hit_off[c0]), -1)
        parts.append(r)
        c0 = c1
    out = {}
    for k in parts[0]:
        if k == "member_off":
            offs, base = [np.zeros(1, np.int64)], 0
            for p in parts:
                offs.append(p[k][1:] + base)
                base += int(p[k][-1])
            out[k] = np.concatenate(offs)
        elif k == "call_counts":
            out[k] = sum(p[k] for p in parts)
        elif k == "call_index":
            continue
        else:
            out[k] = np.concatenate([p[k] for p in parts])
    order = [np.nonzero(out["call"] == c)[0] for c in (2, 1, 0)]
    out["call_index"] = np.concatenate(order).astype(np.int64)
    return out


def main(argv=None):
    args = get_args(argv)
    say("Loading taxonomy.")
    tax = taxonomy.Taxonomy(args.taxonomy)
    say("Initializing contigs.")
    contig_lengths = read_contig_lengths(args.contigs)
    say("Adding gene coordinates.")
    loci = parsers.read_gff_loci(args.gff, device=None if (args.cpu_parse or streamed(args))
                                 else args.device)   # (a streamed run forks its workers: no CUDA in the parent before that)
    analyze(args, tax, contig_lengths, loci)


def analyze(args, tax, contig_lengths, loci, hits=None):
    """Everything after the loci are known: score the contigs and write the outputs.  `loci`: a LocusTable, or for a
    streamed run a streaming.ChunkGenes (each chunk's loci are its own gene calls); `hits`: the parsed blastout if the
    caller already has it (single-call path)."""
    if args.basename is None:
        args.basename = os.path.split(args.contigs)[1].split(".")[0]
    say("Analyzing contigs.")
    if streamed(args):
        from . import streaming
        devices = device_list(args.devices, args.device)
        chunk_bytes = int((args.stream_mb if args.stream_mb > 0 else 256.0) * (1 << 20))
        stats, n_chunks = streaming.run_streaming(
            args, tax, contig_lengths, loci, functools.partial(params_from_args, args),
            devices, max(1, chunk_bytes))
        if not args.quiet:
            for w in sorted(k for k in stats if k != "rest"):
                st = stats[w]
                say("  worker {} on cuda:{}: {:,} contigs / {:,} hits in {} chunk(s) ({:.1f} ms in kernels{})".format(
                    w, st["device"], st["contigs"], st["hits"], st["chunks"], st["ms_kernels"],
                    "; {:,} BGZF members inflated on the device".format(st["inflated_members"])
                    if st.get("inflated_members") else ""))
        say("Finished successfully.")
        return
    if hits is None:
        hits = parsers.read_blast_hits(args.blastout, device=None if args.cpu_parse else args.device)
    if hits.sysmask is None:
        die("more than 32 annotation systems in the subject headers")
    tax.build(hits.distinct_taxa())
    # hits parsed on the GPU: the batch's hit columns are built there from the parser's columns
    pack = packing.pack_resident if gpu_parse.live_resident(hits) is not None else packing.pack
    batch = pack(contig_lengths, loci, hits, tax)
    params = OrgscorerParams.from_args(args, n_systems=len(hits.systems))
    engine = Engine(args.device, params, tax)
    if args.exact_scores:
        engine.set_option("exact", 1)
    if args.write_details:
        # OS:931-937: every clade's gene scores at every evaluated level (the exact pipeline records them)
        res, _ = engine.score_batch_details(batch, download=False)
    else:
        res = score_in_chunks(engine, batch, args.chunk_contigs)
    if not args.quiet:
        st = engine.stats()
        say("  scored {:,} contigs / {:,} hits on cuda:{} ({:.1f} ms in kernels; {:,} contigs on the exact pipeline, "
            "{:,} workspace replays)".format(batch.n_contigs, batch.n_hits, args.device, st["ms_kernels"],
                                             st["fallback_contigs"], st["workspace_retries"]))
    if args.write_details:
        from .streaming import details_order
        writer.write_details_file(os.path.join(args.outdir, args.basename + ".details.tsv.gz"),
                                  engine.details_text(details_order(batch, hits, contig_lengths), batch.contig_names))
    engine.close()
    parsers.close_resident(hits)
    records = writer.build_records(batch, loci, hits, tax, res)
    writer.write_main_output_files(records, args.outdir, args.basename)
    say("Finished successfully.")


if __name__ == "__main__":
    main()
