"""Golden fixture for row a2 (get_reads): outputs of the UNMODIFIED reference BAM_handler::get_reads (compiled into
oracle/_ref/libref_getreads.so over the in-memory htslib stand-in of oracle/stub/sam.h) on seeded synthetic records.
Run in the build container:  python tests/golden/make_golden_getreads.py"""
import os
import sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from pepper_b200 import synth  # noqa: E402
from oracle import oracle  # noqa: E402

SEED, CONTIG, COV, START = 31, 24000, 25, 5000
QUERIES = [(START + 900, START + 2101, False, 0, 0), (START + 10000, START + 11201, False, 0, 0),
           (START - 100, START + 6101, True, 5, 7), (START + 23000, START + 26000, False, 0, 0)]

if __name__ == "__main__":
    oracle.build()
    assert oracle.have_ref_getreads(), "needs oracle/_ref/libref_getreads.so, built from the reference sources"
    rec, _ = synth.simulate_contig_records(CONTIG, COV, synth.ONT, SEED, contig_start=START)
    out = {}
    for qi, (s, e, supp, mq, bq) in enumerate(QUERIES):
        b, pos_end, n_bad = oracle.get_reads(rec, s, e, supp, mq, bq, impl="ref")
        for f in ("pos", "seq_off", "cigar_off", "flags", "mapq", "seq", "qual", "cigar"):
            out[f"q{qi}_{f}"] = getattr(b, f)
        out[f"q{qi}_pos_end"] = pos_end
        out[f"q{qi}_n_bad"] = n_bad
        print(qi, b.n_reads, b.n_bases)
    np.savez_compressed(os.path.join(HERE, "getreads_seed31.npz"), **out)
