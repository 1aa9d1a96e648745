"""`waafle_genecaller` front end over the B200 library: gene calls (GFF) from a waafle_search blastout.

Same positional argument and flags as the reference CLI (waafle/waafle_genecaller.py:44-101), same GFF rows (:217-230,
csv.excel_tab: tab-separated, CRLF line ends).  The per-contig work -- interval sort, overlap links, connected
components, merge (:137-168) -- runs as one CUDA kernel over all contigs (csrc/wfl_genecall.cu): over the columns the
GPU parser keeps on the device (wfl_parser_call_genes), or, with --cpu-parse or a file only the CPU reader takes, over
the host columns (wfl_call_genes).
"""

import argparse
import csv
import ctypes
import os

import numpy as np

from . import parsers
from .engine import EngineError, load_library, mark_cuda_touched
from .utils import say, try_open


def get_args(argv=None):
    parser = argparse.ArgumentParser(
        description="Step 1.5 in the WAAFLE pipeline: use BLAST hits to call genes on contigs (B200-native).",
        formatter_class=argparse.RawTextHelpFormatter)
    parser.add_argument("blastout", help="(custom) blast output from waafle_search")
    parser.add_argument("--gff", default=None, metavar="<path>",
                        help="path for (output) waafle gene calls (.gff)\n[default: <derived from input>]")
    parser.add_argument("--min-overlap", default=0.1, type=float, metavar="<float>")
    parser.add_argument("--min-gene-length", default=200, type=float, metavar="<int>")
    parser.add_argument("--min-scov", default=0.75, type=float, metavar="<float>")
    parser.add_argument("--stranded", action="store_true",
                        help="accepted for compatibility; it has no effect in the reference either\n"
                             "(waafle_genecaller.py:215 compares the flag with the string \"on\")")
    parser.add_argument("--device", type=int, default=0, help="CUDA device index [default: 0]")
    parser.add_argument("--cpu-parse", action="store_true", help="parse the blastout with the CPU reader")
    return parser.parse_args(argv)


def blocks_of(hits):
    """(block offsets [n+1], block names): consecutive runs of one query (iter_contig_hits, utils.py:255-270)."""
    n = len(hits)
    if getattr(hits, "block_starts", None) is not None:
        starts, names = np.asarray(hits.block_starts, dtype=np.int64), list(hits.block_names)
    elif n:
        q = hits.qseqid
        starts = np.flatnonzero(np.r_[True, q[1:] != q[:-1]]).astype(np.int64)
        names = list(q[starts])
    else:
        starts, names = np.zeros(0, np.int64), []
    return np.r_[starts, n].astype(np.int64), names


def call_genes(hits, min_overlap, min_gene_length, min_scov, device=0):
    """Gene calls per contig block: (block names, gene_off [n+1], start, end, strand char codes, kernel ms)."""
    lib = load_library()
    P = ctypes.POINTER
    lib.wfl_call_genes.argtypes = [ctypes.c_int, ctypes.c_int64, P(ctypes.c_int64), P(ctypes.c_int32), P(ctypes.c_int32),
                                   P(ctypes.c_int8), P(ctypes.c_uint8), ctypes.c_double, ctypes.c_double, P(ctypes.c_int32),
                                   P(ctypes.c_int32), P(ctypes.c_int8), P(ctypes.c_int32), P(ctypes.c_float)]
    off, names = blocks_of(hits)
    nb, nh = len(names), len(hits)
    qs = np.ascontiguousarray(hits.qstart, dtype=np.int32)
    qe = np.ascontiguousarray(hits.qend, dtype=np.int32)
    st = np.ascontiguousarray(hits.strand, dtype=np.int8)
    keep = np.ascontiguousarray(np.asarray(hits.scov_modified) >= min_scov, dtype=np.uint8)
    gs, ge, gst = np.zeros(max(nh, 1), np.int32), np.zeros(max(nh, 1), np.int32), np.zeros(max(nh, 1), np.int8)
    gc = np.zeros(max(nb, 1), np.int32)
    ms = ctypes.c_float(0.0)
    ptr = lambda a, t: a.ctypes.data_as(P(t))
    mark_cuda_touched()
    rc = lib.wfl_call_genes(int(device), nb, ptr(off, ctypes.c_int64), ptr(qs, ctypes.c_int32), ptr(qe, ctypes.c_int32),
                            ptr(st, ctypes.c_int8), ptr(keep, ctypes.c_uint8), float(min_overlap), float(min_gene_length),
                            ptr(gs, ctypes.c_int32), ptr(ge, ctypes.c_int32), ptr(gst, ctypes.c_int8), ptr(gc, ctypes.c_int32),
                            ctypes.byref(ms))
    if rc != 0:
        raise EngineError("wfl_call_genes failed with {} (no usable CUDA device? this library has no CPU fallback)".format(rc))
    gc = gc[:nb]
    gene_off = np.zeros(nb + 1, dtype=np.int64)
    np.cumsum(gc, out=gene_off[1:])
    take = np.concatenate([np.arange(off[b], off[b] + gc[b]) for b in range(nb)]) if nb and gene_off[-1] else np.zeros(0, np.int64)
    return names, gene_off, gs[take], ge[take], gst[take], ms.value


def write_gff(path, names, gene_off, start, end, strand):
    with try_open(path, "w") as fh:
        writer = csv.writer(fh, csv.excel_tab)
        for b, contig in enumerate(names):
            for g in range(gene_off[b], gene_off[b + 1]):
                writer.writerow([str(k) for k in (contig, "waafle_genecaller", "gene", int(start[g]), int(end[g]), ".",
                                                  chr(strand[g]), 0, ".")])   # :220-230


def main(argv=None):
    args = get_args(argv)
    if args.gff is None:
        name = os.path.split(args.blastout)[1].split(".")[0]   # utils.path2name / name2path (:201-203)
        args.gff = os.path.join(".", name + ".gff")
    hits, genes = parsers.read_blast_hits_and_genes(args.blastout, args.min_overlap, args.min_gene_length, args.min_scov,
                                                    device=args.device, cpu_parse=args.cpu_parse)
    parsers.close_resident(hits)
    write_gff(args.gff, *genes)
    say("Finished successfully.")


if __name__ == "__main__":
    main()
