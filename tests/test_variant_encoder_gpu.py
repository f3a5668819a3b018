"""GPU parity: CUDA variant encoder (through the C-ABI, host buffers) vs the oracle, bit-exact."""
import os
import numpy as np
import pytest

from pepper_b200 import synth
from tests import kats
from tests.golden import refdigest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def enc():
    from pepper_b200.variant import VariantEncoder
    e = VariantEncoder(0, debug=True)
    yield e
    e.close()


def _compare(oracle, enc, reads, regions, params, name=""):
    want = oracle.variant_encode(reads, regions, params, "port", debug=True)
    got = enc.encode(reads, regions, params)
    # intermediates first: they localise a mismatch
    for r in range(regions.n_regions):
        L1 = int(regions.table[r, 1] - regions.table[r, 0] + 1)
        m, cov, snp, ins, dele = enc.debug_region(r, L1)
        wm, wcov, wsnp, wins, wdel = want["debug"][r]
        assert np.array_equal(cov, wcov), (name, "coverage", np.nonzero(cov != wcov)[0][:10])
        assert np.array_equal(snp, wsnp), (name, "snp_count", np.nonzero(snp != wsnp)[0][:10])
        assert np.array_equal(ins, wins), (name, "insert_count", np.nonzero(ins != wins)[0][:10])
        assert np.array_equal(dele, wdel), (name, "delete_count", np.nonzero(dele != wdel)[0][:10])
        bad = np.argwhere(m != wm)
        assert bad.size == 0, (name, "matrix", bad[:10], m[bad[0][0]], wm[bad[0][0]])
    assert got.keys == want["keys"], (name, got.keys[:10], want["keys"][:10])
    assert np.array_equal(got.positions, want["positions"]), name
    assert np.array_equal(got.depths.astype(np.int32), want["depths"]), name
    assert np.array_equal(got.freqs.astype(np.int32), want["freqs"]), name
    assert np.array_equal(got.region_of, want["region_of"]), name
    wi = oracle.images_to_int8(want["images"])
    bad = np.argwhere(got.images != wi)
    assert bad.size == 0, (name, bad[:10], got.keys[bad[0][0]])
    assert np.array_equal(got.n_per_region, np.bincount(want["region_of"].astype(np.int64), minlength=regions.n_regions))
    return got


@pytest.mark.parametrize("idx", range(12))
def test_kats(oracle_built, enc, idx):
    name, reads, regions, params = kats.variant_kats()[idx]
    _compare(oracle_built, enc, reads, regions, params, name)


@pytest.mark.parametrize("platform,params,seed,nreg,size", [
    (synth.ONT, synth.ont_params(), 3, 2, 6000),
    (synth.HIFI, synth.hifi_params(), 4, 2, 6000),
    (synth.ONT, synth.ont_params(), 5, 5, 20000),
    (synth.ONT, synth.ont_params(), 6, 3, 1537),      # ragged tile tails
])
def test_synthetic(oracle_built, enc, platform, params, seed, nreg, size):
    reads, regions = synth.make_variant_workload(nreg, size, 30, platform, seed=seed)
    got = _compare(oracle_built, enc, reads, regions, params, f"synthetic{seed}")
    assert len(got) > 10


def test_against_compiled_reference(enc):
    """Against the digests of the reference encoder's outputs (tests/golden/refdigest.py) on the same workload."""
    reads, regions = synth.make_variant_workload(2, 8000, 30, synth.ONT, seed=8)
    got = enc.encode(reads, regions, synth.ont_params())
    refdigest.expect("gpu_variant_encoder_seed8", dict(keys=got.keys, positions=got.positions, depths=got.depths, freqs=got.freqs,
                                                       region_of=got.region_of, images_i8=got.images))
    assert np.array_equal(got.n_per_region, np.bincount(got.region_of.astype(np.int64), minlength=regions.n_regions))


def test_ref_with_N_blocks(oracle_built, enc):
    reads, regions = synth.make_variant_workload(2, 4000, 20, synth.ONT, seed=12, n_frac=0.02)
    _compare(oracle_built, enc, reads, regions, synth.ont_params(), "nblocks")


def test_golden(enc):
    g = np.load(os.path.join(GOLD, "variant_ont_seed21.npz"))
    reads, regions = synth.make_variant_workload(2, 5000, 30, synth.ONT, seed=21)
    got = enc.encode(reads, regions, synth.ont_params())
    assert np.array_equal(got.images, g["images"])
    assert np.array_equal(got.positions, g["positions"])
    assert got.keys == [k.decode() for k in g["keys"]]
    assert np.array_equal(got.depths, g["depths"].astype(np.uint8))
    assert np.array_equal(got.freqs, g["freqs"].astype(np.uint8))


def test_empty_and_small(oracle_built, enc):
    # region without reads, region with only mapq-0 reads, one-position region
    ref = "ACGTACGTAC"
    tab = np.array([[100, 109, 100, 109, 0, 10, 0, 0], [200, 209, 200, 209, 0, 10, 0, 1], [300, 300, 300, 300, 0, 1, 1, 2]],
                   dtype=np.int64)
    regions = synth.RegionTable(tab, np.frombuffer(ref.encode(), dtype=np.uint8).copy())
    reads = synth.make_batch([dict(pos=200, seq="TTTTTTTTTT", qual=30, cigar=[(0, 10)], mapq=0),
                              dict(pos=300, seq="T", qual=30, cigar=[(0, 1)])])
    got = _compare(oracle_built, enc, reads, regions, kats.LOOSE, "empty")
    assert got.keys == ["1T"]


def test_capacity_retry(enc):
    reads, regions = synth.make_variant_workload(1, 4000, 30, synth.ONT, seed=2)
    a = enc.encode(reads, regions, synth.ont_params(), capacity=3)
    b = enc.encode(reads, regions, synth.ont_params())
    assert len(a) == len(b) > 3 and np.array_equal(a.images, b.images)


def test_properties_full_size(enc):
    """Size-independent properties at a BASELINE-sized region (100 kb + 2x100): sortedness of the output,
    window/matrix consistency and idempotence (two runs bit-identical)."""
    reads, regions = synth.make_variant_workload(2, 100000, 30, synth.ONT, seed=77)
    a = enc.encode(reads, regions, synth.ont_params())
    b = enc.encode(reads, regions, synth.ont_params())
    assert np.array_equal(a.images, b.images) and a.keys == b.keys
    order = list(zip(a.region_of.tolist(), a.positions.tolist(), a.keys))
    assert order == sorted(order)
    # col 0 of the middle row is the reference code of the candidate position
    ref = regions.ref
    for i in np.linspace(0, len(a) - 1, 200).astype(int):
        r = a.region_of[i]
        x = a.positions[i] - regions.table[r, 0]
        code = {65: 1, 67: 2, 71: 3, 84: 4}.get(int(ref[regions.table[r, 4] + x]), 5)
        assert a.images[i, 16, 0] == code
    assert 500 < len(a) < 20000


def test_more_reads_than_one_list_round(oracle_built, enc):
    """> 1024 reads in one region: k_tile_count scans the region's reads in several rounds (LIST_CAP);
    also a very deep pileup (coverage ~ 390) with mixed indels."""
    rng = np.random.default_rng(99)
    ref = "".join("ACGT"[i] for i in rng.integers(0, 4, 1800))
    S = 5000
    reads = []
    for k in range(2600):
        a = int(rng.integers(0, 1500))
        n = int(rng.integers(120, 300))
        # recurrent variant sites so that the site thresholds are reached: SNPs at x % 50 == 7 (40 % of the reads),
        # a 2-base deletion after x % 120 == 60 (35 %), an insertion after x % 170 == 85 (35 %)
        seq, cig, run = [], [], 0
        x = a
        while x < a + n:
            base = ref[x]
            if x % 50 == 7 and rng.random() < 0.4:
                base = "ACGT"[("ACGT".index(base) + 1 + int(rng.integers(0, 2))) % 4]
            seq.append(base); run += 1
            if x % 120 == 60 and x + 3 < a + n and rng.random() < 0.35:
                cig += [(0, run), (2, 2)]; run = 0; x += 2
            elif x % 170 == 85 and x + 1 < a + n and rng.random() < 0.35:
                ins = ["AC", "A", "ACG"][int(rng.integers(0, 3))]
                cig += [(0, run), (1, len(ins))]; run = 0; seq.extend(ins)
            x += 1
        if run:
            cig.append((0, run))
        seq = "".join(seq)
        reads.append(dict(pos=S + a, seq=seq, qual=[int(q) for q in rng.integers(1, 40, len(seq))], cigar=cig,
                          reverse=bool(rng.random() < 0.5), mapq=int(60 if rng.random() > 0.02 else 0)))
    reads.sort(key=lambda r: r["pos"])
    batch = synth.make_batch(reads)
    tab = np.array([[S, S + 1799, S + 100, S + 1700, 0, 1800, 0, len(reads)]], dtype=np.int64)
    regions = synth.RegionTable(tab, np.frombuffer(ref.encode(), dtype=np.uint8).copy())
    got = _compare(oracle_built, enc, batch, regions, synth.ont_params(), "deep")
    assert len(got) > 40 and {k[0] for k in got.keys} == {"1", "2", "3"}
    assert got.depths.max() == 125            # clamped depth
