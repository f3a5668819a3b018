"""GPU parity: CUDA polish encoder (C-ABI, host buffers) vs the oracle, bit-exact."""
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
    from pepper_b200.polish import PolishEncoder
    e = PolishEncoder(0)
    yield e
    e.close()


def _compare(oracle, enc, reads, regions, name=""):
    want = oracle.polish_encode(reads, regions, "port")
    got = enc.encode(reads, regions)
    assert np.array_equal(got.col_off, want["col_off"]), name
    assert np.array_equal(got.pos, want["pos"]), name
    assert np.array_equal(got.idx, want["idx"]), name
    bad = np.argwhere(got.image != want["image"])
    assert bad.size == 0, (name, bad[:10], got.image[bad[0][0]], want["image"][bad[0][0]])
    return got


@pytest.mark.parametrize("idx", range(4))
def test_kats(oracle_built, enc, idx):
    name, reads, regions = kats.polish_kats()[idx]
    _compare(oracle_built, enc, reads, regions, name)


@pytest.mark.parametrize("platform,seed,nreg,cov", [(synth.ONT, 9, 4, 40), (synth.HIFI, 10, 3, 35), (synth.ONT, 11, 50, 30)])
def test_synthetic(oracle_built, enc, platform, seed, nreg, cov):
    reads, regions = synth.make_polish_workload(nreg, cov, platform, seed=seed)
    got = _compare(oracle_built, enc, reads, regions, f"synthetic{seed}")
    assert got.image.shape[0] > 1000 * nreg


def test_against_compiled_reference(enc):
    """Against the digests of the reference encoder's outputs (tests/golden/refdigest.py) on the same workload."""
    reads, regions = synth.make_polish_workload(5, 40, synth.ONT, seed=13)
    got = enc.encode(reads, regions)
    refdigest.expect("gpu_polish_encoder_seed13", dict(image=got.image, pos=got.pos, idx=got.idx, col_off=got.col_off))


def test_golden(enc):
    g = np.load(os.path.join(GOLD, "polish_ont_seed22.npz"))
    reads, regions = synth.make_polish_workload(3, 40, synth.ONT, seed=22)
    got = enc.encode(reads, regions)
    assert np.array_equal(got.image, g["image"]) and np.array_equal(got.pos, g["pos"])
    assert np.array_equal(got.idx, g["idx"]) and np.array_equal(got.col_off, g["col_off"])


def test_empty_region_and_capacity(oracle_built, enc):
    tab = np.array([[100, 150, 100, 150, 0, 0, 0, 0], [200, 260, 200, 260, 0, 0, 0, 1]], dtype=np.int64)
    regions = synth.RegionTable(tab, np.zeros(1, np.uint8))
    reads = synth.make_batch([dict(pos=190, seq="ACGT" * 20, qual=30, cigar=[(0, 40), (1, 5), (0, 35)])])
    got = _compare(oracle_built, enc, reads, regions, "empty")
    assert got.col_off[1] == 51
    small = enc.encode(reads, regions, capacity=4)
    assert np.array_equal(small.image, got.image)


def test_chunking_matches_reference_rule(enc):
    from pepper_b200.polish import chunk_images
    reads, regions = synth.make_polish_workload(3, 40, synth.ONT, seed=5)
    s = enc.encode(reads, regions)
    imgs, pos, idx, cids, regs = chunk_images(s)
    assert imgs.shape[1:] == (1000, 10)
    for r in range(3):
        n = int(s.col_off[r + 1] - s.col_off[r])
        mine = np.nonzero(regs == r)[0]
        assert list(cids[mine]) == list(range(len(mine)))
        # first chunk = first 1000 columns; second starts 50 columns before the first one's end
        assert np.array_equal(imgs[mine[0]][:min(n, 1000)], s.image[s.col_off[r]:s.col_off[r] + min(n, 1000)])
        if n > 1000:
            assert np.array_equal(pos[mine[1]][:50], s.pos[s.col_off[r] + 950:s.col_off[r] + 1000])
        last = mine[-1]
        pad = np.nonzero(pos[last] == -1)[0]
        assert (imgs[last][pad] == 0).all()


def test_more_reads_than_one_list_round(oracle_built, enc):
    rng = np.random.default_rng(98)
    S = 100
    reads = []
    for k in range(2300):
        a = int(rng.integers(0, 900)); n = int(rng.integers(80, 200))
        seq = "".join("ACGTN"[i] for i in rng.integers(0, 5, n))
        if rng.random() < 0.3:
            p = n // 2
            reads.append(dict(pos=S + a, seq=seq, qual=20, cigar=[(0, p), (1, 3), (0, n - p - 3)], reverse=bool(k % 2)))
        elif rng.random() < 0.3:
            p = n // 2
            reads.append(dict(pos=S + a, seq=seq, qual=20, cigar=[(0, p), (2, 4), (0, n - p)], reverse=bool(k % 2)))
        else:
            reads.append(dict(pos=S + a, seq=seq, qual=20, cigar=[(0, n)], reverse=bool(k % 2), mapq=int(k % 50 != 0) * 60))
    reads.sort(key=lambda r: r["pos"])
    tab = np.array([[S, S + 1100, S, S + 1100, 0, 0, 0, len(reads)]], dtype=np.int64)
    _compare(oracle_built, enc, synth.make_batch(reads), synth.RegionTable(tab, np.zeros(1, np.uint8)), "deep")
