"""Writes reference_digests.json (tests/golden/refdigest.py): the UNMODIFIED reference code compiled into oracle/_ref
(oracle/Makefile, from the reference sources) run on the inputs of every test that compares with it, and the reference's
store readers run on the stores of tests/test_datastore_reference_readers.py.
    python tests/golden/make_golden_digests.py [PATH_OF_THE_REFERENCE_SOURCES]"""
import json
import multiprocessing as mp
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from pepper_b200 import synth  # noqa: E402
from oracle import oracle  # noqa: E402
from tests import kats  # noqa: E402
from tests.golden import refdigest  # noqa: E402


def variant(reads, regions, params):
    return refdigest.variant_fields(oracle.variant_encode(reads, regions, params, "ref"), oracle.images_to_int8)


def _region_100(r):
    reads, regions = synth.make_variant_workload(100, 100000, 30, synth.ONT, seed=103)
    sub, tab = synth.region_batch(reads, regions, r)
    w = oracle.variant_encode(sub, tab, synth.ont_params(), "ref")
    return w["keys"], w["positions"], w["depths"], w["freqs"], oracle.images_to_int8(w["images"])


def encoder_cases(out):
    for idx, (name, reads, regions, params) in enumerate(kats.variant_kats()):
        out["variant_kat_%d" % idx] = variant(reads, regions, params)
    for platform, params, seed in [(synth.ONT, synth.ont_params(), 3), (synth.HIFI, synth.hifi_params(), 4)]:
        out["variant_synthetic_seed%d" % seed] = variant(*synth.make_variant_workload(2, 6000, 30, platform, seed=seed), params)
    for idx, (name, reads, regions) in enumerate(kats.polish_kats()):
        out["polish_kat_%d" % idx] = oracle.polish_encode(reads, regions, "ref")
    out["polish_synthetic_seed9"] = oracle.polish_encode(*synth.make_polish_workload(4, 40, synth.ONT, seed=9), "ref")
    # GPU tests
    out["gpu_variant_encoder_seed8"] = variant(*synth.make_variant_workload(2, 8000, 30, synth.ONT, seed=8), synth.ont_params())
    out["gpu_polish_encoder_seed13"] = oracle.polish_encode(*synth.make_polish_workload(5, 40, synth.ONT, seed=13), "ref")
    for platform, params, cov, seed in [(synth.ONT, synth.ont_params(), 30, 101), (synth.HIFI, synth.hifi_params(), 35, 102)]:
        out["gpu_full_size_seed%d" % seed] = variant(*synth.make_variant_workload(4, 100000, cov, platform, seed=seed), params)
    # 100 regions, one at a time as the reference runs them (test_100_full_size_regions_cross_group_boundary)
    with mp.get_context("spawn").Pool(min(16, os.cpu_count() or 1)) as pool:
        parts = pool.map(_region_100, range(100), chunksize=1)
    out["gpu_full_size_100_regions_seed103"] = dict(
        keys=[k for p in parts for k in p[0]], positions=np.concatenate([p[1] for p in parts]),
        depths=np.concatenate([p[2] for p in parts]), freqs=np.concatenate([p[3] for p in parts]),
        region_of=np.concatenate([np.full(len(p[0]), r, np.int32) for r, p in enumerate(parts)]),
        images_i8=np.concatenate([p[4] for p in parts]))


def getreads_cases(out):
    from tests.test_oracle_getreads import synthetic_queries
    for name, rec, queries in kats.getreads_kats():
        for qi, q in enumerate(queries):
            out["getreads_kat_%s_%d" % (name, qi)] = refdigest.reads_fields(*oracle.get_reads(rec, *q, impl="ref"))
    for seed, platform in [(3, synth.ONT), (4, synth.HIFI)]:
        rec, _ = synth.simulate_contig_records(20000, 15, platform, seed, contig_start=7000)
        for qi, q in enumerate(synthetic_queries(seed)):
            out["getreads_synthetic_seed%d_%d" % (seed, qi)] = refdigest.reads_fields(*oracle.get_reads(rec, *q, impl="ref"))


def realign_cases(out):
    from tests.test_oracle_realign import ssw_cases, realign_workload, realign_fields
    for t, (q, ref) in enumerate(ssw_cases(1, 250)):
        out["ssw_%d" % t] = dict(result=list(oracle.ssw_align(q, ref, "ref")))
    reads, regions = realign_workload()
    for r in range(regions.n_regions):
        row = regions.table[r]
        ref = regions.ref[int(row[4]):int(row[4] + row[5])].tobytes().decode()
        out["realign_r%d" % r] = realign_fields(oracle.realign(reads, int(row[6]), int(row[7]), int(row[0]), int(row[1]) + 20, ref, impl="ref"))
        out["realign_r%d_start300" % r] = realign_fields(
            oracle.realign(reads, int(row[6]), int(row[7]), int(row[0]) + 300, int(row[1]) + 20, ref[300:], impl="ref"))


if __name__ == "__main__":
    oracle.build()
    assert oracle.have_ref() and oracle.have_ref_getreads() and oracle.have_ref_realign(), \
        "needs oracle/_ref, built from the reference sources (make -C oracle REF=...)"
    from tests.golden import make_golden_stores
    fields = {}
    encoder_cases(fields)
    getreads_cases(fields)
    realign_cases(fields)
    table = {case: refdigest.digests(f) for case, f in fields.items()}
    table.update(make_golden_stores.reader_digests(sys.argv[1] if len(sys.argv) > 1 else os.environ.get("PEPPER_REFERENCE", "")))
    with open(refdigest.PATH, "w") as f:
        json.dump(table, f, indent=0, sort_keys=True)
        f.write("\n")
    print("%d cases" % len(table))
