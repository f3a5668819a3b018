"""CPU tests for row a2 (BAM_handler::get_reads): the plain-C restatement (oracle/port_getreads.c) against the UNMODIFIED
reference function compiled into oracle/_ref/libref_getreads.so, on the branch KATs and on seeded synthetic contigs (through
the digests of its outputs, tests/golden/refdigest.py); against the committed golden fixture; and the reservoir sampler
against the reference's literal loop."""
import os
import numpy as np
import pytest

from pepper_b200 import synth
from pepper_b200.reads import reservoir_select, RANDOM_SEED
from tests import kats
from tests.golden import make_golden_getreads as gold, refdigest

GOLD = os.path.join(os.path.dirname(__file__), "golden", "getreads_seed31.npz")
FIELDS = ("pos", "seq_off", "cigar_off", "flags", "mapq", "seq", "qual", "cigar")


def synthetic_queries(seed):
    """25 seeded get_reads queries over the synthetic contig of test_getreads_synthetic_port_vs_reference."""
    start = 7000
    rng = np.random.default_rng(seed)
    for _ in range(25):
        s = int(rng.integers(start - 500, start + 20500))
        e = s + int(rng.choice([1, 2, 50, 1201, 6000]))
        yield s, e, bool(rng.integers(0, 2)), int(rng.choice([0, 0, 10])), int(rng.choice([0, 7]))


def test_getreads_kats_port_vs_reference(oracle_built):
    for name, rec, queries in kats.getreads_kats():
        kept_any = 0
        for qi, q in enumerate(queries):
            a, ae, ab = oracle_built.get_reads(rec, *q, impl="port")
            refdigest.expect("getreads_kat_%s_%d" % (name, qi), refdigest.reads_fields(a, ae, ab))
            kept_any += a.n_reads
        assert kept_any > 20


def test_getreads_kat_expectations(oracle_built):
    """Hand-checked facts about the branch KAT, independent of either implementation's internals."""
    name, rec, queries = kats.getreads_kats()[0]
    a, pos_end, n_bad = oracle_built.get_reads(rec, 160, 260, False, 0, 0, impl="port")
    # first record ("plain match", pos 100, 200M): trimmed to [160, 260] inclusive -> 101 bases, one op
    assert a.pos[0] == 160 and a.seq_off[1] - a.seq_off[0] == 101 and a.cigar[a.cigar_off[0]] == (101 << 4 | 0)
    assert pos_end[0] == 261
    # flag-filtered records never appear (5 records), low MAPQ only with min_mapq
    pos_set = {int(p) for p in a.pos}
    assert not pos_set & {190, 191, 192, 193, 194}
    assert 195 in pos_set
    b, _, _ = oracle_built.get_reads(rec, 160, 260, False, 20, 0, impl="port")
    assert 195 not in {int(p) for p in b.pos}
    c, _, _ = oracle_built.get_reads(rec, 160, 260, True, 0, 0, impl="port")
    assert 194 in {int(p) for p in c.pos}                      # supplementary kept on request
    # record 231: 30M ends exactly at stop; the insertion at stop+1 and everything after are cut
    i = int(np.nonzero(a.pos == 231)[0][0])
    assert a.seq_off[i + 1] - a.seq_off[i] == 30 and a.cigar_off[i + 1] - a.cigar_off[i] == 1 and pos_end[i] == 261
    # record 205 (8I 30M): the leading insertion has no anchor -> dropped, read starts on the match
    i = int(np.nonzero(a.pos == 205)[0][0])
    assert a.cigar[a.cigar_off[i]] == (30 << 4 | 0) and a.seq_off[i + 1] - a.seq_off[i] == 30
    # the record that touches the query only with its deletion keeps no base and is dropped: 18 records, 5 flag-filtered,
    # pos 260/261 not returned by the iterator (end-exclusive), the deletion-only one dropped, the CIGAR-less one dropped
    assert a.n_reads == 18 - 5 - 2 - 1 - 1


@pytest.mark.parametrize("seed,platform", [(3, synth.ONT), (4, synth.HIFI)])
def test_getreads_synthetic_port_vs_reference(oracle_built, seed, platform):
    rec, _ = synth.simulate_contig_records(20000, 15, platform, seed, contig_start=7000)
    total = 0
    for qi, q in enumerate(synthetic_queries(seed)):
        a, ae, ab = oracle_built.get_reads(rec, *q, impl="port")
        refdigest.expect("getreads_synthetic_seed%d_%d" % (seed, qi), refdigest.reads_fields(a, ae, ab))
        total += a.n_reads
    assert total > 50


def test_getreads_port_vs_golden(oracle_built):
    g = np.load(GOLD)
    rec, _ = synth.simulate_contig_records(gold.CONTIG, gold.COV, synth.ONT, gold.SEED, contig_start=gold.START)
    for qi, (s, e, supp, mq, bq) in enumerate(gold.QUERIES):
        a, ae, ab = oracle_built.get_reads(rec, s, e, supp, mq, bq, impl="port")
        for f in FIELDS:
            assert np.array_equal(getattr(a, f), g[f"q{qi}_{f}"]), (qi, f)
        assert np.array_equal(ae, g[f"q{qi}_pos_end"]) and np.array_equal(ab, g[f"q{qi}_n_bad"])
        assert a.n_reads > 10


def test_trimmed_reads_start_on_match(oracle_built):
    """What the encoders rely on (DESIGN §1): every read get_reads returns starts with a match op at its pos."""
    rec, _ = synth.simulate_contig_records(15000, 20, synth.ONT, 9, contig_start=100)
    a, _, _ = oracle_built.get_reads(rec, 3000, 4201, False, 0, 0, impl="port")
    first = a.cigar[a.cigar_off[:-1]] & 15
    assert np.isin(first, [0, 7, 8]).all() and (a.pos >= 3000).all()


@pytest.mark.parametrize("total,allowed", [(10, 10), (11, 10), (4000, 1500), (37, 5), (5, 0)])
def test_reservoir_select_is_the_reference_loop(total, allowed):
    """pepper_variant AlignmentSummarizer.py:113-125 restated literally on indices."""
    got = reservoir_select(total, allowed)
    if total <= allowed:
        assert got is None
        return
    random = np.random.RandomState(RANDOM_SEED)
    sample = []
    for i, read in enumerate(range(total)):
        if len(sample) < allowed:
            sample.append(read)
        else:
            j = random.randint(0, i + 1)
            if j < allowed:
                sample[j] = read
    assert got.tolist() == sample
