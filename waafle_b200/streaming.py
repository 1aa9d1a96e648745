"""Streaming, multi-GPU drive of the orgscorer engine (SURVEY 7.2 step 8 / BASELINE configs[4]).

The reference holds every contig, hit and output row in memory and scores one contig after the other
(waafle/waafle_orgscorer.py:905-960).  Contigs are independent (:943-960) and the blastout is grouped by query
(waafle/utils.py:255-258), so a run of any size is cut into contig-aligned byte ranges of the blastout file:

    parent   scan_blast_chunks()            byte ranges that start where the query name changes
    workers  one process per GPU            read a range -> parse it on the GPU -> pack with the contigs' loci -> Engine.score_batch
                                            -> rows -> per-chunk TSV shards (sorted by contig name)
    parent   merge_shards()                 k-way merge of the shards by contig name (:838) under ONE header whose
                                            annotation columns are the union over all chunks (:824-831)

The engine, the packer and the row builder are the ones of the single-call path (orgscorer.main); the outputs are
byte-identical to it (tests/test_streaming.py on CPU for the merge, tests/test_cli_gpu.py on the GPU end to end).
"""

import heapq
import os

import numpy as np

from . import packing, parsers, writer
from .utils import die, say, write_row

WINDOW = 1 << 20


# ---------------------------------------------------------------------------------------------------------------
# contig-aligned chunks of a blastout file
# ---------------------------------------------------------------------------------------------------------------

def _first_query_change(buf, carry_name):
    """Offset in `buf` (which starts at a row start) of the first row whose query differs from the row before it
    (`carry_name`: query of the row just before `buf`, or None).  -1 if there is none in the complete rows of `buf`."""
    pos, prev = 0, carry_name
    while True:
        nl = buf.find(b"\n", pos)
        if nl < 0:
            return -1, prev
        tab = buf.find(b"\t", pos, nl)
        name = buf[pos:tab if tab >= 0 else nl]
        if prev is not None and name != prev and nl > pos:
            return pos, prev
        if nl > pos:
            prev = name
        pos = nl + 1


def scan_blast_chunks(path, target_bytes):
    """[(offset, length)] covering the file; every range but the first starts at a row whose query name differs from the
    previous row's, and ranges are ~target_bytes long (a single contig's block is never split)."""
    with open(path, "rb") as fh:
        return scan_text_chunks(fh, os.path.getsize(path), target_bytes)


def scan_text_chunks(fh, size, target_bytes):
    """scan_blast_chunks over any seekable reader `fh` of `size` bytes of blastout text (a file, compressed.BgzfReader)."""
    chunks, start = [], 0
    while start < size:
        want = start + target_bytes
        if want >= size:
            chunks.append((start, size - start))
            break
        # row start at or after `want`
        fh.seek(want - 1)
        buf = fh.read(WINDOW)
        nl = buf.find(b"\n")
        while nl < 0 and len(buf) < size - want + 1:
            more = fh.read(WINDOW)
            if not more:
                break
            buf += more
            nl = buf.find(b"\n")
        if nl < 0:
            chunks.append((start, size - start))
            break
        row0 = want - 1 + nl + 1          # absolute offset of a row start
        # query of the row before row0
        back = min(row0 - start, WINDOW)
        fh.seek(row0 - back)
        tail = fh.read(back)
        prev_start = tail.rfind(b"\n", 0, len(tail) - 1) + 1
        prev_row = tail[prev_start:]
        tab = prev_row.find(b"\t")
        carry = prev_row[:tab] if tab >= 0 else prev_row.rstrip(b"\n")
        # first change of query at or after row0
        fh.seek(row0)
        pos_abs, cut = row0, -1
        while pos_abs < size:
            buf = fh.read(WINDOW)
            if not buf:
                break
            last_nl = buf.rfind(b"\n")
            if last_nl < 0:
                more = fh.read(WINDOW)
                while more and b"\n" not in more:
                    buf += more
                    more = fh.read(WINDOW)
                buf += more
                last_nl = buf.rfind(b"\n")
                if last_nl < 0:
                    break
            body = buf[:last_nl + 1]
            off, carry = _first_query_change(body, carry)
            if off >= 0:
                cut = pos_abs + off
                break
            pos_abs += len(body)
            fh.seek(pos_abs)
        if cut < 0 or cut >= size:
            chunks.append((start, size - start))
            break
        chunks.append((start, cut - start))
        start = cut
    return chunks


def _text_cut(buf, target_bytes):
    """Offset in `buf` (text from a row start) of the first query change at or after target_bytes, or -1 when the
    complete rows of `buf` hold none."""
    nl = buf.find(b"\n", max(target_bytes, 1) - 1)
    if nl < 0:
        return -1
    row0 = nl + 1
    prev_row = bytes(buf[buf.rfind(b"\n", 0, nl) + 1:nl])
    tab = prev_row.find(b"\t")
    off, _ = _first_query_change(bytes(buf[row0:]), prev_row[:tab] if tab >= 0 else prev_row)
    return row0 + off if off >= 0 else -1


def stream_text_chunks(path, target_bytes):
    """The text of a generic gzip or bzip2 blastout, inflated as a stream (zlib and bz2 release the GIL), in pieces of
    about target_bytes that start where the query name changes (the rule of scan_blast_chunks)."""
    import bz2
    import gzip
    buf, eof = bytearray(), False
    with (bz2.open if path.endswith(".bz2") else gzip.open)(path, "rb") as fh:
        while True:
            cut = _text_cut(buf, target_bytes) if len(buf) > target_bytes else -1
            if cut > 0:
                yield bytes(buf[:cut])
                del buf[:cut]
            elif eof:
                if buf:
                    yield bytes(buf)
                return
            else:
                more = fh.read(max(WINDOW, target_bytes // 4))
                buf += more
                eof = not more


# ---------------------------------------------------------------------------------------------------------------
# loci by contig, built once
# ---------------------------------------------------------------------------------------------------------------

class LociIndex:
    """Rows of a LocusTable grouped by contig (file order kept inside a contig): the streaming packer looks up the loci
    of a chunk's contigs instead of scanning the whole GFF per chunk."""

    def __init__(self, loci, contig_lengths):
        import pandas as pd
        self.loci = loci
        codes, uniq = pd.factorize(np.asarray(loci.seqname, dtype=object)) if len(loci) else (np.zeros(0, np.int64), [])
        self.order = np.argsort(codes, kind="stable")
        self.off = np.zeros(len(uniq) + 1, dtype=np.int64)
        if len(loci):
            np.cumsum(np.bincount(codes, minlength=len(uniq)), out=self.off[1:])
        self.slot = {nm: k for k, nm in enumerate(uniq)}
        for nm in uniq:
            if nm not in contig_lengths:
                say("  Unknown contig in <{}> file".format("gff"), nm)   # OS:921-923

    def rows(self, names):
        parts = []
        for nm in names:
            k = self.slot.get(nm)
            if k is not None:
                parts.append(self.order[self.off[k]:self.off[k + 1]])
        return np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)

    def subset(self, names):
        """(LocusTable of the contigs' loci, their row numbers in the full table)."""
        rows = self.rows(names)
        lt = self.loci
        sub = parsers.LocusTable.__new__(parsers.LocusTable)
        sub.seqname, sub.start, sub.end = lt.seqname[rows], lt.start[rows], lt.end[rows]
        sub.strand_str, sub.strand = lt.strand_str[rows], lt.strand[rows]
        return sub, rows


class ChunkGenes:
    """Loci of every chunk = the chunk's own waafle_genecaller gene calls (in place of a LociIndex).  Chunks never split a
    contig block, so per-chunk gene calls are the whole file's; contigs without hits have no genes.  With `gff`, every
    chunk also writes its calls as a GFF shard and the run concatenates them there in chunk (= blastout) order."""

    def __init__(self, min_overlap, min_gene_length, min_scov, gff=None):
        self.thresholds = (min_overlap, min_gene_length, min_scov)
        self.gff = gff
        self.loci = parsers.LocusTable([], [], [], [])   # what the contigs without hits are scored against

    def subset(self, names):
        return self.loci, np.zeros(0, dtype=np.int64)


def concat_gff_shards(paths, out):
    """The GFF shards of the chunks, in chunk order, as one file."""
    import shutil
    with open(out, "wb") as dst:
        for path in paths:
            with open(path, "rb") as src:
                shutil.copyfileobj(src, dst)


def chunk_contigs(hits, contig_lengths):
    """Names of the contigs a parsed chunk holds hits for (block order), known or not."""
    if getattr(hits, "block_names", None) is not None:
        return list(hits.block_names)
    q = hits.qseqid
    if len(q) == 0:
        return []
    starts = np.r_[True, q[1:] != q[:-1]]
    return list(q[starts])


def details_order(batch, hits, contig_lengths):
    """Indices of the batch's contigs in blastout order: the row order of the details table (OS:944)."""
    index = {nm: k for k, nm in enumerate(batch.contig_names)}
    return [index[nm] for nm in dict.fromkeys(chunk_contigs(hits, contig_lengths)) if nm in index]


def pack_chunk(names, contig_lengths, loci_index, hits, tax, pack=packing.pack):
    """`pack` (packing.pack or packing.pack_resident) restricted to the contigs `names` (FASTA-known ones); loci rows
    refer to the FULL locus table."""
    known = [nm for nm in dict.fromkeys(names) if nm in contig_lengths]
    sub_lengths = {nm: contig_lengths[nm] for nm in known}
    sub_loci, rows = loci_index.subset(known)
    batch = pack(sub_lengths, sub_loci, hits, tax)
    batch.locus_row = rows[batch.locus_row] if len(rows) else batch.locus_row
    return batch


# ---------------------------------------------------------------------------------------------------------------
# shards and their merge
# ---------------------------------------------------------------------------------------------------------------

SHARD_SEP = "\x1f"   # shard rows: name, number of retained loci, annotation cells follow the fixed cells


def write_shard(records, prefix):
    """Rows of one chunk, sorted by contig name, as <prefix>.<call>.shard files.  First line: the chunk's annotation
    systems; every row: contig name, number of retained loci, the formatted fixed cells, then one cell per system."""
    systems = sorted({s for r in records for d in r["annotations"] for s in d})
    handles = {opt: open("{}.{}.shard".format(prefix, opt), "w") for opt in writer.FORMATS}
    for fh in handles.values():
        fh.write(SHARD_SEP.join(systems) + "\n")
    for r in sorted(records, key=lambda r: r["contig_name"]):
        opt = r["call"]
        cells = [writer.format_field(r[f]) for f in writer.FORMATS[opt]]
        ann = [writer.format_field("|".join(d.get(s, writer.C_MISSING_ANNOTATION) for d in r["annotations"])) for s in systems]
        handles[opt].write(SHARD_SEP.join([r["contig_name"], str(len(r["annotations"]))] + cells + ann) + "\n")
    for fh in handles.values():
        fh.close()
    return systems


def _shard_rows(path, n_fixed, all_systems):
    """(name, row cells) of one shard in name order; the annotation cells are laid out for the run-wide system list."""
    with open(path) as fh:
        head = fh.readline().rstrip("\n")
        systems = head.split(SHARD_SEP) if head else []
        same = systems == all_systems
        for line in fh:
            parts = line.rstrip("\n").split(SHARD_SEP)
            if same:   # the common case: every chunk saw the same systems
                yield parts[0], parts[2:]
                continue
            n_loci = int(parts[1])
            ann = dict(zip(systems, parts[2 + n_fixed:]))
            missing = writer.format_field("|".join([writer.C_MISSING_ANNOTATION] * n_loci))
            yield parts[0], parts[2:2 + n_fixed] + [ann.get(s, missing) for s in all_systems]


def shard_systems(prefixes):
    out = set()
    for p in prefixes:
        with open("{}.{}.shard".format(p, "lgt")) as fh:
            head = fh.readline().rstrip("\n")
            out.update(head.split(SHARD_SEP) if head else [])
    return sorted(out)


def merge_shards(prefixes, outdir, basename, remove=True):
    """k-way merge of the chunk shards by contig name into <basename>.{lgt,no_lgt,unclassified}.tsv (OS:814-894): one
    header with the union of the transferred annotation systems; a system a chunk never saw prints `None` per locus."""
    say("Initializing outputs.")
    systems = shard_systems(prefixes)
    for opt, fmt in writer.FORMATS.items():
        with open(os.path.join(outdir, ".".join([basename, opt, "tsv"])), "w") as out:
            write_row([k.upper() for k in fmt + [writer.C_ANNOTATION_PREFIX + s for s in systems]], out)
            streams = [_shard_rows("{}.{}.shard".format(p, opt), len(fmt), systems) for p in prefixes]
            last = None
            for name, cells in heapq.merge(*streams, key=lambda t: t[0]):
                if name == last:
                    die("blastout is not grouped by query sequence")   # a contig in two chunks
                last = name
                write_row(cells, out)
    if remove:
        for p in prefixes:
            for opt in writer.FORMATS:
                os.remove("{}.{}.shard".format(p, opt))


# ---------------------------------------------------------------------------------------------------------------
# workers
# ---------------------------------------------------------------------------------------------------------------

class ChunkScorer:
    """Everything one device needs to turn a piece of blastout text into shard rows."""

    def __init__(self, device, args, tax, contig_lengths, loci_index, params_factory, cpu_parse=False, engine_factory=None):
        if engine_factory is None:
            from .engine import Engine
            engine_factory = Engine
        self.device, self.args, self.tax = device, args, tax
        self.contig_lengths, self.loci_index = contig_lengths, loci_index
        self.params_factory = params_factory
        self.cpu_parse = cpu_parse
        self.engine = None
        self.Engine = engine_factory   # (device, params, taxonomy) -> object with score_batch / set_params / set_taxonomy / stats / close
        self.parser = None
        self.known_taxa = set()
        self.n_systems = None
        self.stats = dict(contigs=0, hits=0, ms_kernels=0.0, chunks=0, inflated_members=0)

    def parse(self, text, genes=None):
        """The chunk's HitTable; with `genes` = (min_overlap, min_gene_length, min_scov) also its gene calls, as
        (HitTable, (block names, gene_off, start, end, strand))."""
        hits = calls = None
        if not self.cpu_parse:
            from . import gpu_parse
            if self.parser is None:
                self.parser = gpu_parse.BlastParser(self.device)
            hits = self.parser.parse(text)
            if hits is not None and genes is not None:
                calls = (list(hits.block_names) if hits.block_names is not None else [],) + self.parser.call_genes(*genes)
        if hits is None:   # rows the device parser does not reproduce: the CPU reader (reference error behaviour)
            import tempfile
            with tempfile.NamedTemporaryFile(suffix=".blastout", delete=False) as tmp:
                tmp.write(text)
            try:
                hits = parsers.read_blast_hits(tmp.name)
            finally:
                os.remove(tmp.name)
        if genes is None:
            return hits
        if calls is None:
            from . import genecaller
            calls = genecaller.call_genes(hits, *genes, device=self.device)[:5]
        return hits, calls

    def parse_bgzf(self, buf, members, off, length, genes=None):
        """`parse` of text bytes [off, off + length) of a BGZF blastout (bytes `buf`, member table `members`): the members
        that hold them are inflated on the device and only those bytes are parsed.  A member that fails validation on the
        device, or rows the device parser flags, send the chunk to the host (gzip raises its error on a bad member)."""
        import gzip
        from . import compressed
        m0, m1 = compressed.member_range(members, off, length)
        comp, sub = compressed.sub_table(buf, members, m0, m1)
        own = (off - int(members[m0, compressed.OUT_OFF]), length) if m1 > m0 else (0, 0)
        if not self.cpu_parse:
            from . import gpu_parse
            if self.parser is None:
                self.parser = gpu_parse.BlastParser(self.device)
            try:
                hits = self.parser.parse_bgzf(comp, sub, own)
            except gpu_parse.InflateError:
                hits = None
            if hits is not None:
                self.stats["inflated_members"] += len(sub)
                if genes is None:
                    return hits
                names = list(hits.block_names) if hits.block_names is not None else []
                return hits, (names,) + self.parser.call_genes(*genes)
        return self.parse(gzip.decompress(comp)[own[0]:own[0] + own[1]], genes)

    def score(self, names, hits, loci=None, details=None):
        """records of the contigs `names` given their parsed hits (possibly none); `loci`: the chunk's own LocusTable
        (gene calls) instead of the rows of the loci index; `details`: path of the chunk's details shard (rows without
        the header, blastout order) to write."""
        if hits.sysmask is None:
            die("more than 32 annotation systems in the subject headers")
        taxa = hits.distinct_taxa()
        if self.tax.index is None or not taxa <= self.known_taxa:
            self.known_taxa |= taxa
            self.tax.build(self.known_taxa)
            tax_changed = True
        else:
            tax_changed = False
        # hits parsed on this worker's GPU: the batch's hit columns are built there from the parser's columns
        from .gpu_parse import live_resident
        pack = packing.pack_resident if live_resident(hits) is not None else packing.pack
        if loci is None:
            batch = pack_chunk(names, self.contig_lengths, self.loci_index, hits, self.tax, pack)
            loci = self.loci_index.loci
        else:
            batch = pack({nm: self.contig_lengths[nm] for nm in dict.fromkeys(names) if nm in self.contig_lengths},
                         loci, hits, self.tax)
        n_sys = len(hits.systems)
        if self.engine is None:
            self.engine = self.Engine(self.device, self.params_factory(n_sys), self.tax)
            if getattr(self.args, "exact_scores", False):
                self.engine.set_option("exact", 1)
        else:
            if n_sys != self.n_systems:
                self.engine.set_params(self.params_factory(n_sys))
            if tax_changed:
                self.engine.set_taxonomy(self.tax)
        self.n_systems = n_sys
        if details is None:
            res = self.engine.score_batch(batch)
        else:
            res, _ = self.engine.score_batch_details(batch, download=False)
            writer.write_details_file(details, self.engine.details_text(details_order(batch, hits, self.contig_lengths),
                                                                        batch.contig_names), header=False)
        st = self.engine.stats()
        self.stats["contigs"] += batch.n_contigs
        self.stats["hits"] += batch.n_hits
        self.stats["ms_kernels"] += st["ms_kernels"]
        self.stats["chunks"] += 1
        return writer.build_records(batch, loci, hits, self.tax, res), batch.contig_names

    def close(self):
        if self.engine is not None:
            self.engine.close()
        if self.parser is not None:
            self.parser.close()


def _worker(wid, device, path, members, tasks, results, shard_dir, args, tax, contig_lengths, loci_index, params_factory,
            engine_factory=None):
    """Tasks (chunk id, offset, length, chunk file): text bytes [offset, offset + length) of the blastout (a text file,
    or the text of a BGZF file when `members` is its member table), or the whole of `chunk file` (a piece of a generic
    gzip / bzip2 blastout the parent inflated; deleted once parsed)."""
    import mmap
    try:
        scorer = ChunkScorer(device, args, tax, contig_lengths, loci_index, params_factory, cpu_parse=args.cpu_parse,
                             engine_factory=engine_factory)
        genes = loci_index.thresholds if isinstance(loci_index, ChunkGenes) else None
        with open(path, "rb") as fh:
            buf = mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ) if members is not None else None
            while True:
                task = tasks.get()
                if task is None:
                    break
                cid, off, length, chunk_file = task
                if chunk_file is not None:
                    with open(chunk_file, "rb") as cf:
                        text = cf.read()
                    os.remove(chunk_file)
                    parsed = scorer.parse(text, genes)
                elif buf is not None:
                    parsed = scorer.parse_bgzf(buf, members, off, length, genes)
                else:
                    fh.seek(off)
                    parsed = scorer.parse(fh.read(length), genes)
                prefix = os.path.join(shard_dir, "chunk{:06d}".format(cid))
                loci = None
                if genes is not None:
                    from . import genecaller
                    hits, calls = parsed
                    loci = parsers.LocusTable.from_blocks(*calls)
                    if loci_index.gff is not None:
                        genecaller.write_gff(prefix + ".gff", *calls)
                else:
                    hits = parsed
                names = chunk_contigs(hits, contig_lengths)
                records, scored = scorer.score(names, hits, loci,
                                               details=prefix + ".details.gz" if args.write_details else None)
                write_shard(records, prefix)
                results.put(("chunk", cid, prefix, list(scored), None))
        results.put(("done", wid, None, None, dict(scorer.stats, device=device)))
        scorer.close()
    except SystemExit as exc:
        results.put(("error", device, None, None, "worker on cuda:{} exited: {}".format(device, exc)))
    except BaseException as exc:   # noqa: B902 -- the parent must hear about every failure
        import traceback
        results.put(("error", device, None, None, traceback.format_exc() or repr(exc)))


class _TextFeeder:
    """Parent-side reader of a generic gzip / bzip2 blastout: a thread inflates it as a stream, writes each piece
    (stream_text_chunks) to a file in the shard directory and queues it as a task.  At most `slots` files exist at once;
    the parent frees a slot when a worker reports the chunk."""

    def __init__(self, path, chunk_bytes, shard_dir, tasks, n_workers):
        import threading
        self.n_chunks, self.error = None, None
        self.slots = threading.Semaphore(2 * n_workers)
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, args=(path, chunk_bytes, shard_dir, tasks, n_workers),
                                        daemon=True)

    def start(self):   # after the workers are forked: a fork must not copy a thread mid-inflate
        self._thread.start()

    def _run(self, path, chunk_bytes, shard_dir, tasks, n_workers):
        n = 0
        try:
            for cid, text in enumerate(stream_text_chunks(path, chunk_bytes)):
                self.slots.acquire()
                if self._stop.is_set():
                    return
                name = os.path.join(shard_dir, "text{:06d}".format(cid))
                with open(name, "wb") as fh:
                    fh.write(text)
                tasks.put((cid, 0, len(text), name))
                n += 1
        except BaseException as exc:   # noqa: B902 -- re-raised in the parent (a corrupt file: gzip's / bz2's error)
            self.error = exc
        finally:
            self.n_chunks = n
            for _ in range(n_workers):
                tasks.put(None)

    def finish(self):
        self._thread.join()
        if self.error is not None:
            raise self.error
        return self.n_chunks

    def stop(self):
        self._stop.set()
        self.slots.release()
        if self._thread.is_alive():
            self._thread.join()


def run_streaming(args, tax, contig_lengths, loci, params_factory, devices, chunk_bytes, engine_factory=None):
    """The whole streamed run: returns (per-worker stats keyed by worker index, plus "rest"; number of chunks).  `loci`: a
    LocusTable, or a ChunkGenes (every chunk is scored against its own gene calls).  `devices`: CUDA device indices, one worker process each.  The
    CLI's parent process never initialises CUDA before this point, so the workers are plain forks sharing the contig /
    loci tables copy-on-write; a caller that already used CUDA in this process gets spawned workers (pickled tables)."""
    import multiprocessing as mp
    import shutil
    import tempfile
    from . import engine as _engine
    from . import compressed
    loci_index = loci if isinstance(loci, ChunkGenes) else LociIndex(loci, contig_lengths)
    fmt, members = compressed.classify(args.blastout)
    chunks = None   # generic gzip / bzip2: cut while a thread inflates the stream (_TextFeeder)
    if fmt == compressed.BGZF:   # chunks of the BGZF text, cut where the query changes; workers inflate on the device
        import mmap
        with open(args.blastout, "rb") as fh, mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ) as buf:
            reader = compressed.BgzfReader(buf, members)
            chunks = scan_text_chunks(reader, reader.size, chunk_bytes)
    elif fmt == compressed.TEXT:
        chunks = scan_blast_chunks(args.blastout, chunk_bytes) if os.path.getsize(args.blastout) > 0 else []
    shard_dir = tempfile.mkdtemp(prefix="wfl_shards_", dir=args.outdir)
    ctx = mp.get_context("spawn" if _engine.cuda_touched() else "fork")
    tasks, results = ctx.Queue(), ctx.Queue()
    feeder, n_chunks = None, None
    if chunks is None:
        feeder = _TextFeeder(args.blastout, chunk_bytes, shard_dir, tasks, len(devices))
    else:
        n_chunks = len(chunks)
        for cid, (off, length) in enumerate(chunks):
            tasks.put((cid, off, length, None))
        for _ in devices:
            tasks.put(None)
    procs = [ctx.Process(target=_worker, args=(w, d, args.blastout, members, tasks, results, shard_dir, args, tax,
                                               contig_lengths, loci_index, params_factory, engine_factory), daemon=True)
             for w, d in enumerate(devices)]
    for p in procs:
        p.start()
    if feeder is not None:
        feeder.start()
    prefixes, seen, stats, done = {}, set(), {}, 0
    try:
        import queue
        while done < len(devices):
            try:
                kind, a, b, c, d = results.get(timeout=5.0)
            except queue.Empty:
                dead = [p for p in procs if not p.is_alive() and p.exitcode not in (0, None)]
                if dead:   # a worker that died without a word (killed, crashed in native code)
                    die("streaming worker exited with code {}".format(dead[0].exitcode))
                continue
            if kind == "error":
                die(d)
            if kind == "done":
                stats[a] = d
                done += 1
                continue
            if feeder is not None:
                feeder.slots.release()
            dup = seen.intersection(c)
            if dup:
                die("blastout is not grouped by query sequence")   # UT:255-258
            seen.update(c)
            prefixes[a] = b
        for p in procs:
            p.join()
        if feeder is not None:
            n_chunks = feeder.finish()
        # contigs without a single hit: scored like the others (unclassified rows with their loci), in the parent's
        # process on the first device -- after the workers are gone
        rest = [nm for nm in contig_lengths if nm not in seen]
        if rest:
            scorer = ChunkScorer(devices[0], args, tax, contig_lengths, loci_index, params_factory, cpu_parse=True,
                                 engine_factory=engine_factory)
            empty = parsers.hits_from_columns(*([[]] * 10))
            step = max(1, int(args.chunk_contigs))
            for k in range(0, len(rest), step):
                records, _ = scorer.score(rest[k:k + step], empty)
                prefix = os.path.join(shard_dir, "rest{:06d}".format(k // step))
                write_shard(records, prefix)
                prefixes[n_chunks + k // step] = prefix
            stats["rest"] = dict(scorer.stats, device=devices[0])
            scorer.close()
        merge_shards([prefixes[k] for k in sorted(prefixes)], args.outdir, args.basename)
        if args.write_details:   # the contigs without hits ("rest") are never evaluated and have no rows (OS:959)
            writer.concat_details_shards(os.path.join(args.outdir, args.basename + ".details.tsv.gz"),
                                         [prefixes[k] + ".details.gz" for k in range(n_chunks)])
        if isinstance(loci_index, ChunkGenes) and loci_index.gff is not None:
            concat_gff_shards([prefixes[k] + ".gff" for k in range(n_chunks)], loci_index.gff)
    finally:
        if feeder is not None:
            feeder.stop()
        for p in procs:
            if p.is_alive():
                p.terminate()
        shutil.rmtree(shard_dir, ignore_errors=True)
    return stats, n_chunks
