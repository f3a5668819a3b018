"""CPU: the four store layouts written by pepper_b200/datastore.py are the ones the reference's OWN reader code reads back —
pepper_variant dataloader_predict.SequenceDataset (a9), pepper dataloader_predict.SequenceDataset (a12), pepper
Stitch.small_chunk_stitch (a14) and pepper_variant CandidateFinder.small_chunk_stitch (a16, which parses
``str(candidates[i])``).  tests/golden/make_golden_stores.py runs those readers on the stores written here, through an
`h5py` stand-in backed by the npz container, and records digests of each store's layout and of what the reader returned
(tests/golden/refdigest.py).  Each test writes its store again and checks that the layout (dataset paths, dtypes, shapes,
contents) is the one the reader read, and that what the reader returned is what the inputs (or the oracle) say.  The
stand-in hands datasets back unchanged, so a wrong dtype (e.g. fixed bytes instead of str) breaks the reference's parsing
exactly as it would under h5py 2.10."""
import numpy as np

from pepper_b200 import datastore as ds
from tests.golden import refdigest

VARIANT_OPTIONS = dict(snp_p_value=0.1, insert_p_value=0.1, delete_p_value=0.1, snp_p_value_in_lc=0.3, insert_p_value_in_lc=0.35,
                       delete_p_value_in_lc=0.25, report_snp_above_freq=0.0, report_indel_above_freq=0.6)


def layout(fname):
    """Dataset path, dtype, shape and content digest of every dataset of a store."""
    d = ds._Store(fname, mode="r", backend="npz").data
    return [[k, d[k].dtype.str, list(d[k].shape), refdigest.digest(d[k])] for k in sorted(d)]


def _s(x):
    """A str stays itself; anything else (e.g. bytes) shows its type."""
    return x if isinstance(x, str) else repr(x)


# ---- a9: variant image store -> pepper_variant dataloader_predict.SequenceDataset
def write_variant_images(f):
    """Writes the store; returns the (contig, position, depth, candidates, frequencies, image) items it must read back as."""
    rng = np.random.default_rng(1)
    imgs = rng.integers(-128, 128, size=(3, 33, 26)).astype(np.int8)
    keys = ["1T", "2ACG", "3" + "ACGT" * 15]
    with ds.VariantImageStore(f, backend="npz") as s:
        s.write_summary("chr20_1000_2000", "chr20", [1001, 1500, 1999], [30, 125, 7], keys, [5, 12, 3], imgs)
    return [("chr20", p, d, [k], [fr], im) for p, d, k, fr, im in zip([1001, 1500, 1999], [30, 125, 7], keys, [5, 12, 3], imgs)]


def variant_items(items, collated_shape):
    return [[_s(c), int(p), int(d), [_s(x) for x in cand], [int(x) for x in np.ravel(fr)], np.asarray(im).dtype.str,
             np.asarray(im).astype(np.int64).tolist()] for c, p, d, cand, fr, im in items] + [list(collated_shape)]


def test_variant_image_store_read_by_reference_dataloader(tmp_path):
    f = str(tmp_path / "img.hdf5")
    items = write_variant_images(f)
    refdigest.expect("store_variant_images", dict(layout=layout(f), reader=variant_items(items, (2, 33, 26))))


# ---- a16: variant prediction store -> pepper_variant CandidateFinder.small_chunk_stitch
def write_variant_predictions(f):
    """Writes the store; returns (genome, positions, depths, keys, freqs, probs) of its candidates."""
    rng = np.random.default_rng(2)
    L = 600
    genome = "".join("ACGT"[i] for i in rng.integers(0, 4, L))
    n = 120
    positions = np.sort(rng.integers(0, L - 8, n))
    keys = []
    for p in positions:
        t = rng.integers(1, 4)
        keys.append("1" + "ACGT"[rng.integers(0, 4)] if t == 1 else ("2" + genome[p] + "AC" if t == 2 else "3" + genome[p:p + 3]))
    depths = rng.integers(4, 60, n); freqs = np.minimum(depths, rng.integers(1, 30, n))
    probs = rng.dirichlet([0.6, 0.5, 0.4], n).astype(np.float32)
    with ds.VariantPredictionStore(f, backend="npz") as s:
        s.write_prediction(0, ["ctg"] * n, positions, depths, keys, freqs, probs)
    return genome, positions, depths, keys, freqs, probs


def candidate_records(margin, deepvariant):
    return [len(margin), [[_s(a[0]), int(a[1]), int(a[2]), _s(a[3]), _s(a[4]), _s(a[5]), int(a[6]), [int(x) for x in a[7]],
                           round(float(a[8]), 9), bool(a[11])] for a in deepvariant]]


def test_variant_prediction_store_read_by_reference_candidate_finder(tmp_path):
    from oracle import find_candidates as ofc
    f = str(tmp_path / "pred.hdf")
    genome, positions, depths, keys, freqs, probs = write_variant_predictions(f)
    want_m, want_d = ofc.select(VARIANT_OPTIONS, "ctg", positions, depths, keys, freqs, probs.astype(np.float64),
                                lambda c, a, b: genome[max(0, a):max(0, b)])
    assert len(want_d) > 20 and len(want_m) > 5               # fixed-bytes candidates would drop every record
    refdigest.expect("store_variant_predictions", dict(layout=layout(f), reader=candidate_records(want_m, want_d)))


# ---- a12: polish image store -> pepper dataloader_predict.SequenceDataset
def write_polish_images(f):
    """Writes the store; returns the (contig, chunk start, chunk end, chunk id, image, position) items it must read back as."""
    img = (np.arange(10000) % 255).astype(np.uint8).reshape(1000, 10)
    with ds.PolishImageStore(f, backend="npz") as s:
        s.write_summary("ctg1", 0, 1100, 1, img, np.arange(1000), np.zeros(1000, np.int64))
    return [("ctg1", 0, 1100, 1, img, np.arange(1000, dtype=np.int64))]


def polish_items(items):
    return [[_s(c), int(cs), int(ce), int(cid), np.asarray(im).astype(np.int64).tolist(), np.asarray(pos).dtype.str]
            for c, cs, ce, cid, im, pos in items]


def test_polish_image_store_read_by_reference_dataloader(tmp_path):
    f = str(tmp_path / "pimg.hdf")
    items = write_polish_images(f)
    refdigest.expect("store_polish_images", dict(layout=layout(f), reader=polish_items(items)))


# ---- a14: polish prediction store -> pepper Stitch.small_chunk_stitch
POLISH_REGIONS = [(0, 1100), (900, 2000)]


def write_polish_predictions(f):
    """Writes the store; returns its images as (region, chunk id, position, index, bases)."""
    rng = np.random.default_rng(3)
    imgs = []
    with ds.PolishPredictionStore(f, backend="npz") as s:
        for r, (a, b) in enumerate(POLISH_REGIONS):
            n = b - a + 1
            start, end, cid = 0, min(n, 1000), 0
            while True:
                pos = np.full(1000, -1, np.int64); idx = np.full(1000, -1, np.int64)
                pos[:end - start] = np.arange(a + start, a + end); idx[:end - start] = 0
                bases = rng.integers(0, 5, 1000).astype(np.uint8)
                s.write_prediction("ctg1", a, b, cid, pos, idx, bases, np.zeros(1000, np.uint8))
                imgs.append((r, cid, pos, idx, bases)); cid += 1
                if end == n:
                    break
                start = end - 50; end = min(n, start + 1000)
    return imgs


def test_polish_prediction_store_read_by_reference_stitch(tmp_path):
    from oracle import stitch as ostitch
    f = str(tmp_path / "ppred.hdf")
    imgs = write_polish_predictions(f)
    want = ostitch.stitch(np.stack([i[4] for i in imgs]), np.stack([i[2] for i in imgs]), np.stack([i[3] for i in imgs]),
                          np.array([i[0] for i in imgs]), np.array([i[1] for i in imgs]), [r[0] for r in POLISH_REGIONS],
                          [r[1] for r in POLISH_REGIONS])
    assert len(want) > 1000
    refdigest.expect("store_polish_predictions", dict(layout=layout(f), reader=want))
