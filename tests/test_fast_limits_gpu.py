"""The fused fast-path kernel (wfl_fast_contigs) at its hard limits, against the C restatement of the reference.

Each limit is a place where the kernel switches representation or hands a contig to another pass: the 32-locus mask
word, 16-bit staged spans and the leaf-plan table, the compact wire format's field widths, u16 hit indices, the
survivor-pair capacities of the three passes, and the guard bands on --range and on the 4-decimal print edge.

Every GPU comparison runs both engine modes (fast: integer / byte outputs bit-exact, crit / rank within 1e-12 and
printed identically; exact: bit-exact) and both wire formats where the compact one can carry the batch, and asserts
the route the fast-mode run took (engine.stats()), so that a fixture meant for the fast kernel cannot pass by going
to the exact pipeline.  Tests without the gpu mark check that each fixture still has its defining property.
"""
import numpy as np
import pytest

import helpers
from oracle import c_oracle

SCORE_RTOL = 1e-12
MODES = (("fast", 0, SCORE_RTOL), ("exact", 1, 0.0))
gpu = pytest.mark.gpu

# two genera of one family; s__A..s__G as in helpers.TAX8
TAX = helpers.TAX8


def params(flags=None, n_systems=0):
    return helpers.params_for(flags or {}, n_systems)


def n_nodes(tax):
    return len(tax.tables()["parent"])


def check(engine, P, tax, batch, ref=None):
    """Both modes, both wire formats against the C restatement; returns (ref, {run: stats}) with runs
    'fast', 'exact' and, if the batch packs, 'fast_packed' / 'exact_packed'."""
    if ref is None:
        ref = c_oracle.score_batch(P, tax, batch)
    wires = [("", batch)]
    if batch.can_pack(n_nodes(tax), P.n_systems):
        wires.append(("_packed", batch.to_packed(P.min_scov)))
    stats = {}
    engine.set_params(P)
    engine.set_taxonomy(tax)
    try:
        for mode, exact, rtol in MODES:
            engine.set_option("exact", exact)
            for suffix, b in wires:
                got = engine.score_batch(b)
                diffs = helpers.compare_results(ref, got, score_rtol=rtol)
                assert not diffs, (mode + suffix, diffs[:4])
                diffs = helpers.compare_printed(ref, got)
                assert not diffs, (mode + suffix, diffs[:4])
                stats[mode + suffix] = engine.stats()
    finally:
        engine.set_option("exact", 0)
    for k, st in stats.items():
        if k.startswith("exact"):
            assert st["smem_contigs"] == 0, k
    return ref, stats


def fast_runs(stats):
    return [v for k, v in stats.items() if k.startswith("fast")]


def assert_route(stats, smem=None, fallback=None, second=None, reasons=None, pairs=None):
    """The fast-mode runs (both wire formats) took the given route."""
    for st in fast_runs(stats):
        got = {k: st[k] for k in ("smem_contigs", "fallback_contigs", "second_pass_contigs", "pairs_scored",
                                   "guard_trips", "refined_groups")}
        got["fallback_reasons"] = st["fallback_reasons"]
        if smem is not None:
            assert st["smem_contigs"] == smem, got
        if fallback is not None:
            assert st["fallback_contigs"] == fallback, got
        if second is not None:
            assert st["second_pass_contigs"] == second, got
        for r, v in (reasons or {}).items():
            assert st["fallback_reasons"][r] == v, (r, got)
        if pairs is not None:
            assert st["pairs_scored"] == pairs, got
        if smem != 0 or fallback != 0:   # (else the whole batch went to the exact pipeline without the fast kernel)
            assert st["smem_contigs"] + st["fallback_contigs"] == st["contigs"], got


def retained(batch, min_len=200):
    """Retained loci per contig (--min-gene-length)."""
    ln = np.abs(batch.locus_end.astype(np.int64) - batch.locus_start) + 1
    keep = ln >= min_len
    return np.array([int(keep[batch.locus_off[c]:batch.locus_off[c + 1]].sum()) for c in range(batch.n_contigs)])


# ---------------------------------------------------------------------------------------------------------------
# 1. the mask word: 30..33 retained loci, the interesting feature on the last one (bit 31 at G = 32)
# ---------------------------------------------------------------------------------------------------------------
FEATURES = ("island", "weak", "annot", "strand")
MASK_FLAGS = [{}, dict(weak_loci="penalize"), dict(weak_loci="assign-unknown"), dict(stranded=True)]


def mask_contig(G, feature, n_short=0):
    """G retained loci of 300 bp (dyadic scores: every gene score is exact in any summation order); with n_short,
    that many 150-bp loci are interleaved (dropped by --min-gene-length) and carry hits of their own.
    The feature sits on the last retained locus:
      island  clade B (s__F) covers only that locus: an LGT island at the last bit;
      weak    s__A scores 0.125 there: ignored / penalised / an Unknown B side, by --weak-loci;
      annot   two equal-scoring annotated hits there, the later one (s__B) must win;
      strand  the locus is on '-'; s__A's hit is '+', s__F's '-': with --stranded only s__F attaches (LGT)."""
    loci, hits = [], []
    short_every = (G // n_short) if n_short else 0
    pos, kept = 1, 0
    while kept < G:
        if n_short and kept % short_every == short_every // 2 and len(loci) - kept == kept // short_every:
            loci.append((pos, pos + 149, "+"))
            hits.append((pos, pos + 149, "s__D", 1.0, 1.0, "+"))
            pos += 250
            continue
        last = kept == G - 1
        strand = "-" if (last and feature == "strand") else "+"
        loci.append((pos, pos + 299, strand))
        a, b = pos, pos + 299
        if not last:
            hits.append((a, b, "s__A", 0.875, 1.0, "+", 0))
        elif feature == "island":
            hits.append((a, b, "s__F", 0.9375, 1.0, "+", 1))
            hits.append((a + 10, b - 10, "s__A", 0.25, 1.0, "+", 1))
        elif feature == "weak":
            hits.append((a, b, "s__A", 0.125, 1.0, "+", 1))
        elif feature == "annot":
            hits.append((a, b, "s__A", 0.875, 1.0, "+", 1))
            hits.append((a + 5, b - 5, "s__C", 0.5, 1.0, "+", 1))
            hits.append((a, b, "s__B", 0.875, 1.0, "+", 1))
        else:
            hits.append((a, b, "s__A", 0.875, 1.0, "+", 1))
            hits.append((a, b, "s__F", 0.9375, 1.0, "-", 1))
        pos += 400
        kept += 1
    return dict(loci=loci, hits=hits)


def mask_batch():
    cs, gs = [], []
    for G in (30, 31, 32, 33):
        for f in FEATURES:
            cs.append(mask_contig(G, f))
            gs.append(G)
    for f in FEATURES:   # 40 raw loci, 8 of them short and interleaved: 32 retained
        cs.append(mask_contig(32, f, n_short=8))
        gs.append(32)
    for f in FEATURES:   # short contigs keep the batch at <= 32 loci per contig (else it all goes to the exact pipeline)
        cs.append(mask_contig(2, f))
        gs.append(2)
    return helpers.make_batch(cs, TAX) + (np.array(gs),)


def boundary_batches():
    """The same four G = 32 contigs, padded once to nl == 32 n (fast kernel) and once to 32 n + 1 (exact pipeline)."""
    base = [mask_contig(32, f) for f in FEATURES]
    pad32 = mask_contig(32, "annot")
    pad33 = mask_contig(33, "annot")
    return helpers.make_batch(base + [pad32], TAX)[0], helpers.make_batch(base + [pad33], TAX)[0], len(base)


def test_mask_fixture_shape():
    batch, tax, gs = mask_batch()
    assert np.array_equal(retained(batch), gs)
    raw = np.diff(batch.locus_off)
    assert np.array_equal(raw[16:20], [40] * 4)
    assert batch.n_loci <= 32 * batch.n_contigs   # the batch is eligible for the fast kernel
    b32, b33, k = boundary_batches()
    assert b32.n_loci == 32 * b32.n_contigs and b33.n_loci == 32 * b33.n_contigs + 1
    assert np.array_equal(retained(b32), [32] * 5)


@gpu
@pytest.mark.parametrize("flags", MASK_FLAGS, ids=["ignore", "penalize", "assign-unknown", "stranded"])
def test_mask_word_vs_c_oracle(engine, flags):
    batch, tax, gs = mask_batch()
    P = params(flags, 1)
    ref, stats = check(engine, P, tax, batch)
    n33 = int((gs == 33).sum())
    assert_route(stats, smem=batch.n_contigs - n33, fallback=n33, reasons={0: n33})
    # the feature on the last retained locus is really decided there
    last = batch.locus_off[1:] - 1
    feat = np.array([f for _ in range(6) for f in FEATURES])
    island, annot, strand = feat == "island", feat == "annot", feat == "strand"
    assert np.array_equal(ref["ann_winner"][last[annot], 0], batch.hit_off[1:][annot] - 1)   # the later s__B hit
    if not flags:
        assert np.all(ref["call"][island] == 2)
        assert np.all(ref["synteny"][last[island]] == ord("B"))
    assert np.all(ref["call"][strand] == (2 if flags.get("stranded") else 1))


@gpu
def test_mask_word_batch_boundary(engine):
    """nl == 32 n: the fast kernel runs; nl == 32 n + 1: the whole batch goes to the exact pipeline.  The shared contigs
    give identical bytes (dyadic scores: the fast path's sums are exact too)."""
    b32, b33, k = boundary_batches()
    tax = helpers.make_batch([mask_contig(32, f) for f in FEATURES], TAX)[1]
    P = params({}, 1)
    _, st32 = check(engine, P, tax, b32)
    _, st33 = check(engine, P, tax, b33)
    assert_route(st32, smem=b32.n_contigs, fallback=0)
    assert_route(st33, smem=0, fallback=0)
    engine.set_params(P)
    engine.set_taxonomy(tax)
    r32, r33 = engine.score_batch(b32), engine.score_batch(b33)
    nl = int(b32.locus_off[k])
    for key in ("call", "direction", "lifts", "clade1", "clade2", "lca", "best1", "best2", "n_members_a"):
        assert np.array_equal(r32[key][:k], r33[key][:k]), key
    for key in ("crit", "rank"):
        assert np.array_equal(r32[key][:k].view(np.int64), r33[key][:k].view(np.int64)), key
    for key in ("synteny", "locus_flags", "ann_winner"):
        assert np.array_equal(r32[key][:nl], r33[key][:nl]), key
    m = int(r32["member_off"][k])
    assert np.array_equal(r32["member_off"][:k + 1], r33["member_off"][:k + 1])
    assert np.array_equal(r32["members"][:m], r33["members"][:m])


# ---------------------------------------------------------------------------------------------------------------
# 2. 16-bit coordinates and the leaf-plan table
# ---------------------------------------------------------------------------------------------------------------
def gene_pair(g1, g2, tail=False):
    """Loci g1 = (start, end), g2 = (start, end): s__A covers g1, s__F covers g2 (an LGT pair)."""
    return dict(loci=[(g1[0], g1[1], "+"), (g2[0], g2[1], "+")],
                hits=[(g1[0], g1[1], "s__A", 0.8, 1.0, "+"), (g2[0], g2[1], "s__F", 0.9375, 1.0, "+"),
                      (g1[0] + 7, g1[1], "s__B", 0.5, 1.0, "-")])


def coord_batches():
    fit = [
        dict(loci=[(64236, 65535, "+"), (60001, 61000, "+")],      # hits ending at 65535
             hits=[(64236, 65535, "s__A", 0.875, 1.0, "+"), (65000, 65535, "s__B", 0.9375, 1.0, "+"),
                   (60001, 61000, "s__A", 0.875, 1.0, "+")]),
        dict(loci=[(1, 1000, "+"), (1101, 2100, "+")],             # a hit with qstart 0
             hits=[(0, 1000, "s__A", 0.875, 1.0, "+"), (1101, 2100, "s__A", 0.875, 1.0, "+"),
                   (0, 300, "s__F", 1.0, 1.0, "+")]),
        gene_pair((1, 16384), (16501, 17500)),                      # the longest gene the plan table holds, at k2
        gene_pair((20001, 20000 + 16384), (1, 1000)),
    ]
    wide = [
        dict(loci=[(64237, 65536, "+"), (60001, 61000, "+")],      # hits ending at 65536
             hits=[(64237, 65536, "s__A", 0.875, 1.0, "+"), (60001, 61000, "s__A", 0.875, 1.0, "+")]),
        gene_pair((1, 16385), (16501, 17500)),                      # one bp past the plan table
        dict(loci=[(1, 70000, "+"), (70101, 71100, "+")],          # 70 kb gene: site slices past 16 bits
             hits=[(1, 70000, "s__A", 0.875, 1.0, "+"), (65600, 69999, "s__F", 1.0, 1.0, "+"),
                   (70101, 71100, "s__F", 0.875, 1.0, "+"), (30000, 70000, "s__D", 0.9375, 1.0, "+")]),
    ]
    edge = [fit[0], wide[0]]   # the two sides of the 16-bit limit alone
    return helpers.make_batch(fit, TAX), helpers.make_batch(wide, TAX), helpers.make_batch(edge[1:], TAX)


def test_coord_fixture_shape():
    (fit, tax), (wide, tax2), (e65536, tax3) = coord_batches()
    assert max(fit.hit_qend.max(), fit.hit_qstart.max()) == 65535 and fit.hit_qstart.min() == 0
    assert fit.can_pack(n_nodes(tax)) and not wide.can_pack(n_nodes(tax2))
    assert int(e65536.hit_qend.max()) == 65536 and not e65536.can_pack(n_nodes(tax3))
    lens = np.abs(fit.locus_end - fit.locus_start) + 1
    assert lens.max() == 16384
    lens = np.abs(wide.locus_end - wide.locus_start) + 1
    assert 16385 in lens and lens.max() == 70000


@gpu
@pytest.mark.parametrize("flags", [{}, dict(weak_loci="assign-unknown"), dict(min_overlap=0.5, stranded=True)])
def test_16bit_coordinates_vs_c_oracle(engine, flags):
    (fit, tax), (wide, tax2), _ = coord_batches()
    P = params(flags)
    ref, stats = check(engine, P, tax, fit)
    assert "fast_packed" in stats
    assert_route(stats, smem=fit.n_contigs, fallback=0)
    ref, stats = check(engine, P, tax2, wide)
    assert "fast_packed" not in stats
    # 65536: staged spans are 16-bit (reason 2); 16385 bp and 70 kb: longer than the plan table (reason 0)
    assert_route(stats, smem=0, fallback=3, reasons={0: 2, 2: 1})


@gpu
def test_plan_table_grows_between_calls():
    """On one engine: a batch whose longest gene is 3000 bp (table at 4096), then one with a 9000-bp gene."""
    from waafle_b200.engine import Engine
    small = [gene_pair((1, n), (n + 101, n + 1100)) for n in (300, 1777, 3000)]
    large = small + [gene_pair((1, 9000), (9101, 10100)), gene_pair((1, 4097), (4201, 5000))]
    P = params({})
    eng = Engine(0)
    try:
        for cs in (small, large):
            batch, tax = helpers.make_batch(cs, TAX)
            _, stats = check(eng, P, tax, batch)
            assert_route(stats, smem=batch.n_contigs, fallback=0)
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------------------------
# 3. compact-format fields: 14-bit taxon index with strand and scov bits, 8-bit system mask
# ---------------------------------------------------------------------------------------------------------------
def big_taxonomy_batch(nodes):
    """A taxonomy of exactly `nodes` nodes; the hits sit on the last node (index nodes - 1), one of them on the minus
    strand and one failing --min-scov."""
    fixed = 6   # r__Root, Unknown, k__B, g__G1, g__G2, s__zz
    edges = [("k__B", "r__Root"), ("g__G1", "k__B"), ("g__G2", "k__B"), ("s__zz", "g__G2")]
    edges += [("s__a{:05d}".format(i), "g__G1") for i in range(nodes - fixed)]
    cs = [
        dict(loci=[(1, 1000, "-"), (1101, 2100, "+")],
             hits=[(1, 1000, "s__zz", 0.875, 1.0, "-"), (1, 1000, "s__zz", 0.9375, 0.5, "-"),
                   (1101, 2100, "s__a00000", 0.875, 1.0, "+"), (1101, 2100, "s__zz", 0.875, 0.74, "+")]),
        dict(loci=[(1, 1000, "+"), (1101, 2100, "-")],
             hits=[(1, 1000, "s__zz", 0.875, 1.0, "-"), (1101, 2100, "s__zz", 0.875, 1.0, "-"),
                   (1, 1000, "s__a00001", 1.0, 0.7, "+"), (1101, 2100, "s__a00001", 0.5, 1.0, "+")]),
    ]
    return helpers.make_batch(cs, edges)


def systems_batch(S):
    """Annotation winners on system bit S - 1 (and bit 0): the last hit attaining the maximum per (locus, system)."""
    top = 1 << (S - 1)
    cs = []
    for k in range(3):
        cs.append(dict(loci=[(1, 1000, "+"), (1101, 2100, "+"), (2201, 3200, "-")],
                       hits=[(1, 1000, "s__A", 0.875, 1.0, "+", top), (1, 1000, "s__B", 0.875, 1.0, "+", top | 1),
                             (1101, 2100, "s__A", 0.9375, 1.0, "+", top), (1101, 2100, "s__D", 0.5, 1.0, "+", top),
                             (1101, 2100, "s__D", 0.25, 1.0, "+", 1), (2201, 3200, "s__A", 0.875, 1.0, "-", 1),
                             (2201, 3200, "s__F", 0.875 + k / 64, 1.0, "+", top)]))
    cs.append(dict(loci=[(1, 1000, "+")], hits=[(1, 1000, "s__A", 0.875, 1.0, "+", 0)]))
    return helpers.make_batch(cs, TAX)


def test_compact_fields_fixture_shape():
    for nodes, packs in ((16384, True), (16385, False)):
        batch, tax = big_taxonomy_batch(nodes)
        assert n_nodes(tax) == nodes and tax.index["s__zz"] == nodes - 1
        assert batch.can_pack(n_nodes(tax)) == packs
    batch, tax = big_taxonomy_batch(16384)
    w = batch.to_packed(0.75)["hit_tax16"]
    assert int(w[0]) == 0x3fff | 0x4000 | 0x8000 and int(w[1]) == 0x3fff | 0x4000
    for S, packs in ((8, True), (9, False), (32, False)):
        batch, tax = systems_batch(S)
        assert int(batch.hit_sysmask.max()) >> (S - 1) == 1
        assert batch.can_pack(n_nodes(tax), S) == packs


@gpu
@pytest.mark.parametrize("flags", [{}, dict(stranded=True), dict(min_scov=0.0)])
def test_taxon_index_16383_packed_vs_wide(engine, flags):
    batch, tax = big_taxonomy_batch(16384)
    P = params(flags)
    ref, stats = check(engine, P, tax, batch)
    assert "fast_packed" in stats
    assert_route(stats, smem=batch.n_contigs, fallback=0)
    assert 16383 in ref["clade1"].tolist() + ref["clade2"].tolist()


@gpu
def test_compact_format_limits_rejected(engine):
    from waafle_b200.engine import EngineError
    batch, tax = big_taxonomy_batch(16385)
    P = params({})
    ref, stats = check(engine, P, tax, batch)   # wide format only
    assert "fast_packed" not in stats
    assert_route(stats, smem=batch.n_contigs, fallback=0)
    with pytest.raises(EngineError):
        engine.score_batch(batch.to_packed(P.min_scov))
    batch, tax = systems_batch(9)
    engine.set_params(params({}, 9))
    engine.set_taxonomy(tax)
    with pytest.raises(EngineError):
        engine.score_batch(batch.to_packed(0.75))


@gpu
@pytest.mark.parametrize("S", [8, 9, 32])
def test_system_bits_vs_c_oracle(engine, S):
    batch, tax = systems_batch(S)
    P = params({}, S)
    ref, stats = check(engine, P, tax, batch)
    assert ("fast_packed" in stats) == (S <= 8)
    assert_route(stats, smem=batch.n_contigs, fallback=0)
    assert (ref["ann_winner"][:, S - 1] >= 0).sum() >= 6


# ---------------------------------------------------------------------------------------------------------------
# 4. contigs with 65 535 and 70 000 hits among ordinary ones
# ---------------------------------------------------------------------------------------------------------------
SPECIES = ["s__A", "s__B", "s__C", "s__D", "s__E", "s__F", "s__G", "t__A1"]


def large_batch(seed=5):
    rng = np.random.default_rng(seed)
    big_cs = []
    for big in (65535, 70000):
        loci = [(1 + 1100 * i, 1000 + 1100 * i, "+-"[i % 2]) for i in range(20)]
        li = rng.integers(0, 20, big)
        a = rng.integers(0, 500, big)
        b = a + rng.integers(300, 500, big)
        tx = rng.integers(0, len(SPECIES), big)
        sc = np.round(rng.uniform(0.3, 1.0, big), 3)
        cv = rng.choice([1.0, 0.9, 0.5], big)
        st = rng.choice(["+", "-"], big)
        hits = [(1 + 1100 * int(i) + int(x), 1 + 1100 * int(i) + int(y), SPECIES[int(t)], float(s), float(c), str(d))
                for i, x, y, t, s, c, d in zip(li, a, b, tx, sc, cv, st)]
        big_cs.append(dict(loci=loci, hits=hits))
    cs = []
    for k in range(300):
        G = 2 + k % 4
        loci = [(1 + 900 * i, 800 + 900 * i, "+") for i in range(G)]
        hits = []
        for i in range(G):
            sp = SPECIES[(k + (i == G - 1) * (k % 3)) % 7]
            hits.append((1 + 900 * i, 800 + 900 * i, sp, float(np.round(rng.uniform(0.6, 1.0), 3)), 1.0, "+"))
            hits.append((50 + 900 * i, 700 + 900 * i, SPECIES[(k + 3) % 7], float(np.round(rng.uniform(0.3, 1.0), 3)), 1.0, "+"))
        cs.append(dict(loci=loci, hits=hits))
    return helpers.make_batch(cs[:50] + big_cs[:1] + cs[50:200] + big_cs[1:] + cs[200:], TAX)


def test_large_fixture_shape():
    batch, tax = large_batch()
    h = np.diff(batch.hit_off)
    assert sorted(h)[-2:] == [65535, 70000]
    assert np.median(h) < 16


@gpu
def test_large_contigs_vs_c_oracle(engine):
    batch, tax = large_batch()
    P = params({})
    ref, stats = check(engine, P, tax, batch)
    # 70 000 hits: more than u16 hit indices hold (reason 1); 65 535 hits: more staged entries than any slice (reason 3,
    # first and second pass); everything else in the fast kernel
    assert_route(stats)
    for st in fast_runs(stats):
        assert st["fallback_reasons"][1] == 1 and st["fallback_reasons"][3] == 2, st["fallback_reasons"]
        # (an ordinary contig may trip a rank guard on a tie of its random scores)
        assert st["fallback_contigs"] == 2 + st["guard_trips"] and st["guard_trips"] <= 3, st


# ---------------------------------------------------------------------------------------------------------------
# 5. two-clade survivor list: exactly a*b pairs pass the mask prefilter
# ---------------------------------------------------------------------------------------------------------------
SURVIVORS = [(8, 8), (5, 13), (32, 32), (25, 41), (32, 64), (3, 683), (45, 46)]


def survivor_batch(a, b, per=3):
    """Clades A_1..A_a each cover locus 0 at >= k2, B_1..B_b locus 1; none covers both, so exactly a*b pairs survive.
    (A_1, B_1) ranks 1.0 and every other pair at most 0.925: the best is unique and no rank sits near --range of it.
    `per` hits per clade (three: the clade table fits the first-pass slice; one: it does not)."""
    edges = [("k__B", "r__Root"), ("g__GA", "k__B"), ("g__GB", "k__B")]
    edges += [("s__A{:04d}".format(i), "g__GA") for i in range(a)] + [("s__B{:04d}".format(j), "g__GB") for j in range(b)]
    hits = []
    for side, m, (lo, hi) in (("A", a, (1, 1000)), ("B", b, (1101, 2100))):
        for i in range(m):
            v = 1.0 if i == 0 else 0.81 + 0.04 * i / m
            for r in range(per):
                hits.append((lo + 3 * r, hi - 2 * r, "s__{}{:04d}".format(side, i), v - 0.001 * r, 1.0, "+"))
    return helpers.make_batch([dict(loci=[(1, 1000, "+"), (1101, 2100, "+")], hits=hits)], edges)


def surviving_pairs(batch, k2=0.8):
    """Pairs of clades whose per-locus maxima cover both loci at k2 (full-length hits: gene score = hit score)."""
    cover = {}
    for t, q1, s in zip(batch.hit_taxon, batch.hit_qstart, batch.hit_score):
        if s >= k2 + 1e-9:
            cover.setdefault(int(t), set()).add(0 if q1 < 1100 else 1)
    cl = sorted(cover)
    return sum(1 for i, x in enumerate(cl) for y in cl[i + 1:] if cover[x] | cover[y] == {0, 1})


@pytest.mark.parametrize("a,b", SURVIVORS)
def test_survivor_fixture_shape(a, b):
    batch, tax = survivor_batch(a, b)
    assert surviving_pairs(batch) == a * b


@gpu
@pytest.mark.parametrize("a,b", SURVIVORS)
def test_survivor_list_capacities(engine, a, b):
    """First pass holds 64 pairs, the 'pairs' pass 1024, the 3x slice 2048; beyond that the exact pipeline.  (3, 683) has
    686 clades and 2058 hits: its 3x slice does not fit shared memory and fit_layout shrinks it (and its pair list)."""
    batch, tax = survivor_batch(a, b)
    ns = a * b
    ref, stats = check(engine, params({}), tax, batch)
    assert ref["call"][0] == 2 and ref["best1"][0] == tax.index["s__A0000"]
    if ns <= 64:
        assert_route(stats, smem=1, fallback=0, second=0, reasons={6: 0}, pairs=ns)
    elif ns <= 1024:
        assert_route(stats, smem=1, fallback=0, second=1, reasons={6: 1}, pairs=ns)
    elif ns <= 2048:
        assert_route(stats, smem=1, fallback=0, second=2, reasons={6: 2}, pairs=ns)
    else:
        assert_route(stats, smem=0, fallback=1, second=2, reasons={6: 3})


@gpu
def test_clade_table_capacity(engine):
    """One hit per clade: 96 clades overflow the first pass's clade table (reason 4); the 3x slice holds them and its
    2048 survivor slots hold the 32 x 64 pairs."""
    batch, tax = survivor_batch(32, 64, per=1)
    ref, stats = check(engine, params({}), tax, batch)
    assert_route(stats, smem=1, fallback=0, second=1, reasons={4: 1, 6: 0}, pairs=2048)


# ---------------------------------------------------------------------------------------------------------------
# 6. guards: the --range edge and the 4-decimal print edge
# ---------------------------------------------------------------------------------------------------------------
def range_batches():
    """One-clade options 0.875 vs 0.625 at --range 0.25, two-clade 1.0 vs 0.9375 at --range 0.0625: exactly on the edge
    and 5e-14 inside it."""
    L0, L1 = (1, 1000), (1101, 2100)
    one = []
    for eps in (0.0, 5e-14, -5e-14):
        one.append(dict(loci=[(*L0, "+"), (*L1, "+")],
                        hits=[(*L0, "s__A", 0.875, 1.0, "+"), (*L1, "s__A", 0.875, 1.0, "+"),
                              (*L0, "s__F", 0.625 + eps, 1.0, "+"), (*L1, "s__F", 0.625 + eps, 1.0, "+")]))
    two = []
    for eps in (0.0, 5e-14, -5e-14):
        two.append(dict(loci=[(*L0, "+"), (*L1, "+")],
                        hits=[(*L0, "s__A", 1.0, 1.0, "+"), (*L1, "s__F", 1.0, 1.0, "+"),
                              (*L1, "s__G", 0.875 + eps, 1.0, "+")]))
    return (helpers.make_batch(one, TAX), dict(range=0.25)), (helpers.make_batch(two, TAX), dict(range=0.0625))


EDGE_VALUES = (0.91235, 0.87665, 0.99995, 0.80005)


def print_edge_batch():
    cs = []
    for n in range(200, 3001, 50):                # one-clade, one gene: crit == rank == mean of n copies of x.xxxx5
        for v in EDGE_VALUES:
            cs.append(dict(loci=[(1, n, "+")], hits=[(1, n, "s__A", v, 1.0, "+")]))
    for n in (300, 777, 1000, 2345):              # ranks that average to a half
        cs.append(dict(loci=[(1, n, "+"), (n + 101, 2 * n + 100, "+")],
                       hits=[(1, n, "s__D", 0.9234, 1.0, "+"), (n + 101, 2 * n + 100, "s__D", 0.9235, 1.0, "+")]))
    for n in (250, 999, 1500, 2999):              # two-clade: crit 0.89255 and rank 0.90245 on edges
        cs.append(dict(loci=[(1, n, "+"), (n + 101, n + 1100, "+")],
                       hits=[(1, n, "s__A", 0.91235, 1.0, "+"), (n + 101, n + 1100, "s__F", 0.89255, 1.0, "+")]))
    return helpers.make_batch(cs, TAX)


def unknown_edge_batch():
    """--weak-loci assign-unknown: the weak locus' Unknown score 1 - 0.08765 is an edge, read off the dense row."""
    cs = []
    for n in (300, 1000, 2718):
        cs.append(dict(loci=[(1, 1000, "+"), (1101, 1100 + n, "+")],
                       hits=[(1, 1000, "s__A", 0.9375, 1.0, "+"), (1101, 1100 + n, "s__B", 0.08765, 1.0, "+")]))
    return helpers.make_batch(cs, TAX)


def edge_contigs(ref):
    cl = np.asarray(ref["call"]) != 0
    return int(sum(1 for c in np.nonzero(cl)[0]
                   if helpers.near_print_edge(ref["crit"][c]) or helpers.near_print_edge(ref["rank"][c])))


def test_guard_fixture_shape():
    (b1, flags1), (b2, flags2) = range_batches()
    ref = c_oracle.score_batch(params(flags1), b1[1], b1[0])
    assert np.all(ref["call"] == 1)
    # the 0.625 option is kept exactly on the edge (d == --range) and 5e-14 inside it, dropped 5e-14 outside
    assert ref["n_members_a"].tolist() == [2, 2, 1]
    ref = c_oracle.score_batch(params(flags2), b2[1], b2[0])
    assert np.all(ref["call"] == 2)
    batch, tax = print_edge_batch()
    ref = c_oracle.score_batch(params({}), tax, batch)
    assert edge_contigs(ref) > 100
    batch, tax = unknown_edge_batch()
    P = params(dict(weak_loci="assign-unknown"))
    ref = c_oracle.score_batch(P, tax, batch)
    assert np.all(ref["call"] == 2) and np.all(ref["clade2"] == tax.index["Unknown"])
    assert edge_contigs(ref) == batch.n_contigs


@gpu
def test_range_edge_guard(engine):
    for (batch, tax), flags in range_batches():
        ref, stats = check(engine, params(flags), tax, batch)
        # every option pair is within 1e-12 of --range from the best: the guard hands them all to the exact pipeline
        assert_route(stats, smem=0, fallback=batch.n_contigs, reasons={7: batch.n_contigs})
        for st in fast_runs(stats):
            assert st["guard_trips"] == batch.n_contigs


@gpu
def test_print_edge_refinement(engine):
    batch, tax = print_edge_batch()
    ref, stats = check(engine, params({}), tax, batch)
    assert_route(stats, smem=batch.n_contigs, fallback=0)
    for st in fast_runs(stats):
        assert st["refined_groups"] >= edge_contigs(ref) and st["guard_trips"] == 0


@gpu
def test_print_edge_on_unknown_row(engine):
    batch, tax = unknown_edge_batch()
    ref, stats = check(engine, params(dict(weak_loci="assign-unknown")), tax, batch)
    assert_route(stats, smem=0, fallback=batch.n_contigs, reasons={7: batch.n_contigs})


# ---------------------------------------------------------------------------------------------------------------
# 7. printed scores of the full-size workloads
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("config,n,flags", [
    ("cfg2", None, {}),
    ("cfg3", 30000, {}),
    ("cfg5", 20000, dict(weak_loci="assign-unknown")),
])
def test_full_size_printed_scores(engine, config, n, flags):
    """The workloads of test_full_size_bit_exact_vs_c_oracle: crit / rank of every classified contig print as the
    C restatement's do, print-edge contigs included."""
    from waafle_b200 import synth
    data = synth.generate_config(config, n_contigs=n, seed=1000, annotations=(config == "cfg5"))
    tax = data.taxonomy()
    batch = data.to_batch(tax)
    P = params(flags, 1 if config == "cfg5" else 0)
    ref = c_oracle.score_batch(P, tax, batch)
    engine.set_params(P)
    engine.set_taxonomy(tax)
    got = engine.score_batch(batch)
    st = engine.stats()
    assert st["smem_contigs"] > 0.9 * batch.n_contigs
    assert not helpers.compare_results(ref, got, score_rtol=SCORE_RTOL)
    diffs = helpers.compare_printed(ref, got)
    assert not diffs, (len(diffs), diffs[:4])
    assert edge_contigs(ref) > 0
    assert st["refined_groups"] > 0


# ---------------------------------------------------------------------------------------------------------------
# 8. wfl_pack_results: the device-packed results equal the numpy packer's, and shards merge to the whole
# ---------------------------------------------------------------------------------------------------------------
def unclassified_batch():
    cs = [dict(loci=[(1, 1000, "+"), (1101, 2100, "+")],
               hits=[(1, 1000, "s__A", 0.25, 1.0, "+"), (1101, 2100, "s__B", 0.125, 1.0, "+")]),
          dict(loci=[(1, 1000, "+")], hits=[]), dict(loci=[], hits=[(1, 500, "s__A", 0.9, 1.0, "+")]),
          dict(loci=[(1, 100, "+")], hits=[(1, 100, "s__A", 0.9, 1.0, "+")])]
    return helpers.make_batch(cs, TAX)


def pack_cases():
    mask, mtax, _ = mask_batch()
    (fit, ftax), _, _ = coord_batches()
    return [("S0", fit, ftax, 0), ("S1_mask", mask, mtax, 1), ("S8", *systems_batch(8), 8), ("S32", *systems_batch(32), 32),
            ("unclassified", *unclassified_batch(), 0), ("n1", fit.slice(2, 3), ftax, 0)]


def test_pack_fixture_shape():
    batch, tax = unclassified_batch()
    ref = c_oracle.score_batch(params({}), tax, batch)
    assert np.all(ref["call"] == 0) and len(ref["members"]) == 0


@gpu
@pytest.mark.parametrize("case", range(6), ids=["S0", "S1_mask", "S8", "S32", "unclassified", "n1"])
def test_pack_results_device_vs_host(engine, case):
    import torch
    from waafle_b200 import dist
    from waafle_b200.engine import unpack_results
    name, batch, tax, S = pack_cases()[case]
    P = params({}, S)
    ref = c_oracle.score_batch(P, tax, batch)
    engine.set_params(P)
    engine.set_taxonomy(tax)

    def device_bytes(b):
        engine.score_batch_device(b)
        blob, stream = dist.device_blob(engine)
        stream.synchronize()
        out = blob.cpu().numpy().copy()
        torch.cuda.synchronize()
        return out

    for exact in (0, 1):
        engine.set_option("exact", exact)
        try:
            dev = device_bytes(batch)
            res = engine.score_batch(batch)
        finally:
            engine.set_option("exact", 0)
        host = dist.pack_results_host(res)
        assert dev.shape == host.shape and np.array_equal(dev, host), (name, exact)
        assert not helpers.compare_results(ref, unpack_results(dev), score_rtol=0.0 if exact else SCORE_RTOL)
    whole = engine.score_batch(batch)
    if batch.n_contigs >= 2:
        cut = batch.n_contigs // 2
        blobs = [device_bytes(batch.slice(0, cut)), device_bytes(batch.slice(cut, batch.n_contigs))]
        merged = dist.merge_blobs(blobs, [0, int(batch.hit_off[cut])])
        assert not helpers.compare_results(whole, merged), name
