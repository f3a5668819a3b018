"""CPU tests: the plain-C restatement (oracle/port_encoders.c) against the UNMODIFIED reference C++
compiled into oracle/_ref, on the hand-written KATs and on seeded synthetic regions (through the digests of its outputs,
tests/golden/refdigest.py); and against the committed golden fixtures (tests/golden/, produced by
tests/golden/make_golden.py from oracle/_ref)."""
import os
import numpy as np
import pytest

from pepper_b200 import synth
from tests import kats
from tests.golden import refdigest

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("idx", range(12))
def test_variant_kat_port_vs_reference(oracle_built, idx):
    name, reads, regions, params = kats.variant_kats()[idx]
    a = oracle_built.variant_encode(reads, regions, params, "port")
    refdigest.expect("variant_kat_%d" % idx, refdigest.variant_fields(a, oracle_built.images_to_int8))
    assert len(a["keys"]) > 0 or name in ("refskip_pad_fallthrough",), name


@pytest.mark.parametrize("platform,params,seed", [(synth.ONT, synth.ont_params(), 3), (synth.HIFI, synth.hifi_params(), 4)])
def test_variant_synthetic_port_vs_reference(oracle_built, platform, params, seed):
    reads, regions = synth.make_variant_workload(2, 6000, 30, platform, seed=seed)
    a = oracle_built.variant_encode(reads, regions, params, "port")
    refdigest.expect("variant_synthetic_seed%d" % seed, refdigest.variant_fields(a, oracle_built.images_to_int8))
    assert len(a["keys"]) > 10


@pytest.mark.parametrize("idx", range(4))
def test_polish_kat_port_vs_reference(oracle_built, idx):
    name, reads, regions = kats.polish_kats()[idx]
    refdigest.expect("polish_kat_%d" % idx, oracle_built.polish_encode(reads, regions, "port"))


def test_polish_wrap_quirk(oracle_built):
    """cov == 0 and three '*' counts -> (3*254) & 255 == 250 (SURVEY §8a a11)."""
    name, reads, regions = kats.polish_kats()[0]
    a = oracle_built.polish_encode(reads, regions, "port")
    col = 125  # inside the deletion (positions 120..129), not its first base
    row = a["image"][col]
    assert row[9] == (2 * 254) & 255 and row[8] == 254   # 2 forward reads, 1 reverse read, coverage 0
    first = a["image"][120]  # first deleted position carries coverage 3*10
    assert first[9] == int((2 / 30) * 254) and first[8] == int((1 / 30) * 254)


def test_polish_synthetic_port_vs_reference(oracle_built):
    reads, regions = synth.make_polish_workload(4, 40, synth.ONT, seed=9)
    refdigest.expect("polish_synthetic_seed9", oracle_built.polish_encode(reads, regions, "port"))


def test_golden_variant(oracle_built):
    g = np.load(os.path.join(GOLD, "variant_ont_seed21.npz"))
    reads, regions = synth.make_variant_workload(2, 5000, 30, synth.ONT, seed=21)
    a = oracle_built.variant_encode(reads, regions, synth.ont_params(), "port")
    assert np.array_equal(oracle_built.images_to_int8(a["images"]), g["images"])
    assert np.array_equal(a["positions"], g["positions"])
    assert np.array_equal(a["depths"], g["depths"]) and np.array_equal(a["freqs"], g["freqs"])
    assert a["keys"] == [k.decode() for k in g["keys"]]


def test_golden_polish(oracle_built):
    g = np.load(os.path.join(GOLD, "polish_ont_seed22.npz"))
    reads, regions = synth.make_polish_workload(3, 40, synth.ONT, seed=22)
    a = oracle_built.polish_encode(reads, regions, "port")
    for k in ("image", "pos", "idx", "col_off"):
        assert np.array_equal(a[k], g[k]), k
