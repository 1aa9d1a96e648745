"""`waafle_genecaller` + `waafle_orgscorer` in one pass: contigs, blastout and taxonomy in, the orgscorer's outputs out,
with no intermediate GFF.

The blastout is read and parsed once (on the GPU unless --cpu-parse); the gene calls run over the hit columns the parser
keeps on the device (wfl_parser_call_genes) and become the loci the contigs are scored against.  The output files are
byte-identical to `python -m waafle_b200.genecaller <blastout> --gff x.gff` followed by `python -m waafle_b200.orgscorer
<contigs> <blastout> x.gff <taxonomy>` with the same values: the orgscorer's flags verbatim, --min-gene-length and
--min-scov shared by both stages (waafle_genecaller.py:81-101, imported by the orgscorer), the genecaller's
--min-overlap as --genecaller-min-overlap.  --gff also writes the gene calls, the bytes the genecaller CLI writes.
"""

import argparse

from . import orgscorer, parsers, taxonomy
from .genecaller import write_gff
from .utils import read_contig_lengths, say


def get_args(argv=None):
    parser = argparse.ArgumentParser(
        description="Steps 1.5 and 2 in the WAAFLE pipeline in one pass: call genes on contigs from the blast hits and "
                    "identify contigs best explained by one clade vs. a pair of clades (putative LGT), without an "
                    "intermediate GFF.  B200-native engine.",
        formatter_class=argparse.RawTextHelpFormatter)
    g = parser.add_argument_group("required inputs")
    g.add_argument("contigs", help="contigs file (.fasta format)")
    g.add_argument("blastout", help="output of waafle_search for one set of contigs (.blastout)")
    g.add_argument("taxonomy", help="taxonomy file for the blast database used to make <blastout>")
    g = parser.add_argument_group("gene calls (waafle_genecaller)")
    g.add_argument("--gff", default=None, metavar="<path>",
                   help="also write the gene calls to this path (.gff) [default: not written]")
    g.add_argument("--genecaller-min-overlap", default=0.1, type=float, metavar="<float>",
                   help="the genecaller's --min-overlap: hits that overlap by this fraction of the shorter one are merged\n"
                        "into one gene [default: 0.1]; --min-overlap is the orgscorer's hit/gene overlap")
    orgscorer.add_flags(parser)
    return parser.parse_args(argv)


def gene_thresholds(args):
    """(min_overlap, min_gene_length, min_scov) of the gene calls."""
    return args.genecaller_min_overlap, args.min_gene_length, args.min_scov


def main(argv=None):
    args = get_args(argv)
    say("Loading taxonomy.")
    tax = taxonomy.Taxonomy(args.taxonomy)
    say("Initializing contigs.")
    contig_lengths = read_contig_lengths(args.contigs)
    if orgscorer.streamed(args):
        # the workers call the genes of their own chunks (no CUDA in this process before they are forked)
        from . import streaming
        orgscorer.analyze(args, tax, contig_lengths, streaming.ChunkGenes(*gene_thresholds(args), gff=args.gff))
        return
    say("Calling genes.")
    hits, genes = parsers.read_blast_hits_and_genes(args.blastout, *gene_thresholds(args), device=args.device,
                                                    cpu_parse=args.cpu_parse)
    if args.gff is not None:
        write_gff(args.gff, *genes)
    orgscorer.analyze(args, tax, contig_lengths, parsers.LocusTable.from_blocks(*genes), hits)


if __name__ == "__main__":
    main()
