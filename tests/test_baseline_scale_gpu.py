"""GPU parity at BASELINE.json's own sizes (VERDICT r1 item 1): full 100 kb intervals (+2 x 100 bp halo = 100,201
positions per region, pepper_variant ImageGenerationUI.py:307-316) compared with the UNMODIFIED reference encoder
compiled into oracle/_ref (through the digests of its outputs, tests/golden/refdigest.py) and with the plain-C port, for
the ONT and HiFi presets, and one batch of 100 distinct regions through the public host-buffer call so that the region-group pipelining of
pb_variant_call_host (first group 24, then 96 regions) and its capacity retry cross a group boundary.  Network outputs
of the shipped (tcgen05) mode are compared with oracle/nets.py for the candidates of sampled regions."""
import numpy as np
import pytest

from pepper_b200 import synth
from tests.golden import refdigest

pytestmark = pytest.mark.gpu
TOL = 1e-3
MARGIN = 1e-4


def _fields(calls):
    return dict(keys=calls.keys, positions=calls.positions, depths=calls.depths, freqs=calls.freqs, region_of=calls.region_of,
                images_i8=calls.images)


def _same_candidates(got, want, oracle, images=True):
    assert got.keys == want["keys"]
    assert np.array_equal(got.positions, want["positions"])
    assert np.array_equal(got.depths.astype(np.int32), want["depths"])
    assert np.array_equal(got.freqs.astype(np.int32), want["freqs"])
    assert np.array_equal(got.region_of, want["region_of"])
    if images:
        assert np.array_equal(got.images, oracle.images_to_int8(want["images"]))


@pytest.mark.parametrize("platform,params,cov,seed", [
    (synth.ONT, synth.ont_params(), 30, 101),
    (synth.HIFI, synth.hifi_params(), 35, 102),
])
def test_full_size_regions_vs_reference(oracle_built, platform, params, cov, seed):
    """4 full-size regions per preset, encoder bit-exact against the compiled reference; network (default mode) against
    the PyTorch oracle on every candidate of those regions."""
    from oracle import nets
    from pepper_b200.pipeline import VariantCaller
    reads, regions = synth.make_variant_workload(4, 100000, cov, platform, seed=seed)
    assert int(regions.table[0, 1] - regions.table[0, 0] + 1) == 100201
    state = nets.make_variant_weights(seed)
    caller = VariantCaller(state)
    calls = caller.call(reads, regions, params, want_images=True)
    want = oracle_built.variant_encode(reads, regions, params, "port")
    _same_candidates(calls, want, oracle_built)
    refdigest.expect("gpu_full_size_seed%d" % seed, _fields(calls))
    assert len(calls) > (1000 if platform is synth.ONT else 100)
    probs = nets.variant_predict(state, calls.images, threads=16)
    assert np.abs(probs - calls.probs).max() < TOL, np.abs(probs - calls.probs).max()
    srt = np.sort(probs, axis=1)
    clear = (srt[:, -1] - srt[:, -2]) > MARGIN
    assert np.array_equal(calls.probs.argmax(1)[clear], probs.argmax(1)[clear])
    caller.close()


def test_100_full_size_regions_cross_group_boundary(oracle_built):
    """100 distinct full-size ONT regions in ONE host call: 3 staged groups (24 + 76 ...), network over whole 9,472-candidate
    chunks of the accumulated candidates, capacity retry in the middle of the call."""
    from oracle import nets
    from pepper_b200.pipeline import VariantCaller
    n_regions = 100
    reads, regions = synth.make_variant_workload(n_regions, 100000, 30, synth.ONT, seed=103)
    params = synth.ont_params()
    state = nets.make_variant_weights(3)
    caller = VariantCaller(state)
    calls = caller.call(reads, regions, params, want_images=True)
    # the oracle one region at a time (that is how the reference runs: one RegionalSummaryGenerator per interval)
    off = 0
    for r in range(n_regions):
        sub, tab = synth.region_batch(reads, regions, r)
        w = oracle_built.variant_encode(sub, tab, params, "port")
        n = len(w["keys"])
        sl = slice(off, off + n)
        assert calls.keys[off:off + n] == w["keys"], r
        assert np.array_equal(calls.positions[sl], w["positions"]), r
        assert np.array_equal(calls.depths[sl].astype(np.int32), w["depths"]), r
        assert np.array_equal(calls.freqs[sl].astype(np.int32), w["freqs"]), r
        assert np.all(calls.region_of[sl] == r), r
        assert np.array_equal(calls.images[sl], oracle_built.images_to_int8(w["images"])), r
        off += n
    assert off == len(calls) > 9472 * 3
    refdigest.expect("gpu_full_size_100_regions_seed103", _fields(calls))
    # capacity far too small: the retry happens inside the second group and must give the same answer
    small = caller.call(reads, regions, params, capacity=40000)
    assert np.array_equal(small.probs, calls.probs) and np.array_equal(small.positions, calls.positions)
    # network: candidates of three sampled regions (first group, group boundary, last) against the PyTorch oracle
    counts = np.bincount(calls.region_of, minlength=n_regions)
    starts = np.concatenate([[0], np.cumsum(counts)])
    for r in (0, 24, n_regions - 1):
        sl = slice(int(starts[r]), int(starts[r + 1]))
        probs = nets.variant_predict(state, calls.images[sl], threads=16)
        assert np.abs(probs - calls.probs[sl]).max() < TOL
        srt = np.sort(probs, axis=1)
        clear = (srt[:, -1] - srt[:, -2]) > MARGIN
        assert np.array_equal(calls.probs[sl].argmax(1)[clear], probs.argmax(1)[clear])
    caller.close()
