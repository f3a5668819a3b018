"""CPU tests for row f1: the plain-C restatement of the reference realigner (oracle/port_realign.c) against the UNMODIFIED
reference sources (simple_aligner.cpp + ssw_cpp.cpp + ssw.c compiled into oracle/_ref/libref_realign.so) through the
digests of their outputs (tests/golden/refdigest.py), and against a committed golden fixture made from them
(tests/golden/make_golden_realign.py)."""
import os
import numpy as np

from pepper_b200 import synth
from tests.golden import refdigest

GOLD = os.path.join(os.path.dirname(__file__), "golden", "realign_seed41.npz")


def _mutate(rng, s, sub, ins, dele):
    out = []
    for ch in s:
        u = rng.random()
        if u < dele:
            continue
        out.append("ACGT"[rng.integers(0, 4)] if u < dele + sub else ch)
        while rng.random() < ins:
            out.append("ACGT"[rng.integers(0, 4)])
    return "".join(out)


def ssw_cases(seed, n):
    rng = np.random.default_rng(seed)
    for t in range(n):
        L = int(rng.choice([5, 20, 40, 62, 63, 64, 70, 100, 300, 700]))
        ref = "".join("ACGT"[i] for i in rng.integers(0, 4, L + int(rng.integers(0, 60))))
        st = int(rng.integers(0, max(1, len(ref) - L + 1)))
        q = _mutate(rng, ref[st:st + L], *((0.02, 0.02, 0.02) if t % 3 else (0.1, 0.08, 0.08)))
        if t % 7 == 0:
            q = "".join("ACGT"[i] for i in rng.integers(0, 4, 10)) + q
        if t % 11 == 0:
            ref = ref[:len(ref) // 2] + "NNN" + ref[len(ref) // 2 + 3:]
        if t % 13 == 0:
            q = q[:len(q) // 2] + "".join("ACGT"[i] for i in rng.integers(0, 4, int(rng.integers(8, 30)))) + q[len(q) // 2:]
        if t % 17 == 0:
            q = q[:len(q) // 3] + q[len(q) // 3 + int(rng.integers(8, 30)):]
        if q:
            yield q, ref


def test_ssw_port_vs_reference(oracle_built):
    n = 0
    for q, ref in ssw_cases(1, 250):
        refdigest.expect("ssw_%d" % n, dict(result=list(oracle_built.ssw_align(q, ref, "port"))))
        n += 1
    assert n > 200


def test_ssw_known_answers(oracle_built):
    """Hand-checkable alignments (match 4, mismatch 6, gap open 8, extend 2)."""
    a = oracle_built.ssw_align("ACGTACGTTGCAACGTTGCATTTACG", "GGGACGTACGTTGCAACGTTGCATTTACGCCC", "port")
    assert a == (104, 3, 28, 0, 25, 0, "26=")
    # one mismatch in the middle: 25 matches - 6
    a = oracle_built.ssw_align("ACGTACGTTGCAAGGTTGCATTTACG", "ACGTACGTTGCAACGTTGCATTTACG", "port")
    assert a[0] == 25 * 4 - 6 and a[6] == "13=1X12="
    # a 3-base deletion from the read: 8 + 2*2 = 12 penalty
    ref = "ACGGTCATTGCAAGCTTAGGCATCGATTACAGGCATTCAGGA"
    q = ref[:20] + ref[23:]
    a = oracle_built.ssw_align(q, ref, "port")
    assert a[0] == len(q) * 4 - 12 and "3D" in a[6]


def realign_workload():
    """The seeded polish workload of test_realign_port_vs_reference."""
    from pepper_b200.realign import realign_regions
    reads, regions = synth.make_polish_workload(2, 12, synth.ONT, seed=7)
    return reads, realign_regions(regions, synth.make_reference(2 * 1000 + 1, 7))


def realign_fields(out):
    return dict(zip(("pos", "pos_end", "cigar_off", "cigar"), out))


def test_realign_port_vs_reference(oracle_built):
    reads, regions = realign_workload()
    for r in range(regions.n_regions):
        row = regions.table[r]
        ref = regions.ref[int(row[4]):int(row[4] + row[5])].tobytes().decode()
        a = oracle_built.realign(reads, int(row[6]), int(row[7]), int(row[0]), int(row[1]) + 20, ref, impl="port")
        refdigest.expect("realign_r%d" % r, realign_fields(a))
        # reads that start before the region start are dropped by both
        a = oracle_built.realign(reads, int(row[6]), int(row[7]), int(row[0]) + 300, int(row[1]) + 20, ref[300:], impl="port")
        assert a[0].shape[0] < int(row[7] - row[6])
        refdigest.expect("realign_r%d_start300" % r, realign_fields(a))


def test_realign_port_vs_golden(oracle_built):
    from tests.golden import make_golden_realign as gold
    g = np.load(GOLD)
    reads, regions = gold.workload()
    for r in range(regions.n_regions):
        row = regions.table[r]
        ref = regions.ref[int(row[4]):int(row[4] + row[5])].tobytes().decode()
        pos, pos_end, co, cig = oracle_built.realign(reads, int(row[6]), int(row[7]), int(row[0]), int(row[1]) + 20, ref, impl="port")
        assert np.array_equal(pos, g[f"r{r}_pos"]) and np.array_equal(pos_end, g[f"r{r}_pos_end"])
        assert np.array_equal(co, g[f"r{r}_cigar_off"]) and np.array_equal(cig, g[f"r{r}_cigar"])
