"""Runs the reference's OWN store readers (pepper_variant dataloader_predict.SequenceDataset, pepper
dataloader_predict.SequenceDataset, pepper Stitch.small_chunk_stitch, pepper_variant CandidateFinder.small_chunk_stitch)
on the stores written by tests/test_datastore_reference_readers.py and returns the digests of each store's layout and of
what the reader returned (tests/golden/refdigest.py), for make_golden_digests.py.  The readers are imported from the
reference sources with stand-in modules: an `h5py` backed by the npz container (h5py / libhdf5 are not required) that hands
datasets back unchanged, torchvision, the compiled `build` modules, and `np.int = int` (alias removed from numpy >= 1.24)."""
import os
import sys
import tempfile
import types

import numpy as np

from tests import test_datastore_reference_readers as t
from tests.golden import refdigest


class _Leaf:
    def __init__(self, a):
        self.a = a

    def __getitem__(self, k):
        if k != ():
            return self.a[k]
        return self.a[()] if self.a.shape == () else self.a


class _Node:
    def __init__(self, store, prefix):
        self.s, self.p = store, prefix

    def keys(self):
        return self.s.keys(self.p) if self.p else sorted({k.split("/", 1)[0] for k in self.s.data})

    def __contains__(self, k):
        return k in self.keys()

    def __getitem__(self, k):
        path = (self.p + "/" + k).strip("/")
        return _Leaf(self.s.data[path]) if path in self.s.data else _Node(self.s, path)


def _install_standins(ref_path):
    from pepper_b200 import datastore as ds

    class _File(_Node):
        def __init__(self, name, mode="r"):
            super().__init__(ds._Store(name, mode="r", backend="npz"), "")

        def __enter__(self):
            return self

        def __exit__(self, *a):
            pass

        def close(self):
            pass
    h5 = types.ModuleType("h5py"); h5.File = _File
    tv = types.ModuleType("torchvision"); tvt = types.ModuleType("torchvision.transforms")
    tvt.Compose = lambda x: x; tvt.ToTensor = lambda: None; tv.transforms = tvt
    pv = types.ModuleType("pepper_variant.build.PEPPER_VARIANT")

    class CandidateImagePrediction:
        def __init__(self, contig, position, depth, candidates, candidate_frequency, prediction_base, prediction_type):
            self.contig, self.position, self.depth = contig, position, depth
            self.candidates, self.candidate_frequency = candidates, candidate_frequency
            self.prediction_base, self.prediction_type = prediction_base, prediction_type
    pv.CandidateImagePrediction = CandidateImagePrediction
    bv = types.ModuleType("pepper_variant.build"); bv.PEPPER_VARIANT = pv
    bp = types.ModuleType("pepper.build"); bp.PEPPER = types.ModuleType("pepper.build.PEPPER")
    sys.modules.update({"h5py": h5, "torchvision": tv, "torchvision.transforms": tvt, "pepper_variant.build": bv,
                        "pepper_variant.build.PEPPER_VARIANT": pv, "pepper.build": bp, "pepper.build.PEPPER": bp.PEPPER})
    sys.path.insert(0, ref_path)
    np.int = int
    return pv


def reader_digests(ref_path):
    assert os.path.isdir(os.path.join(ref_path, "pepper_variant")), "pass the path of the reference sources"
    pv = _install_standins(ref_path)
    from pepper_variant.modules.python.models.dataloader_predict import SequenceDataset as VariantDataset
    from pepper_variant.modules.python import CandidateFinder as RefCF
    from pepper.modules.python.models.dataloader_predict import SequenceDataset as PolishDataset
    from pepper.modules.python import Stitch as RefStitch
    out = {}
    d = tempfile.mkdtemp()

    f = os.path.join(d, "img.hdf5")
    t.write_variant_images(f)
    data = VariantDataset(None, input_file=f)
    items = [data[i] for i in range(len(data))]
    batch = VariantDataset.my_collate([data[0], data[1]])
    out["store_variant_images"] = dict(layout=t.layout(f), reader=t.variant_items(items, tuple(batch[5].shape)))

    f = os.path.join(d, "pred.hdf")
    genome = t.write_variant_predictions(f)[0]

    class FASTA_handler:
        def __init__(self, path):
            pass

        def get_reference_sequence(self, contig, a, b):
            return genome[max(0, a):max(0, b)]
    pv.FASTA_handler = FASTA_handler
    got_m, got_d = RefCF.small_chunk_stitch(types.SimpleNamespace(fasta="x", **t.VARIANT_OPTIONS), [(f, "batch_0")])
    out["store_variant_predictions"] = dict(layout=t.layout(f), reader=t.candidate_records(got_m, got_d))

    f = os.path.join(d, "pimg.hdf")
    t.write_polish_images(f)
    data = PolishDataset(None, file_list=[f])
    items = [tuple(data[i])[:6] for i in range(len(data))]
    out["store_polish_images"] = dict(layout=t.layout(f), reader=t.polish_items(items))

    f = os.path.join(d, "ppred.hdf")
    t.write_polish_predictions(f)
    first, last, seq = RefStitch.small_chunk_stitch("ctg1", [(f, "ctg1", a, b) for a, b in t.POLISH_REGIONS])
    out["store_polish_predictions"] = dict(layout=t.layout(f), reader=seq)
    return {case: refdigest.digests(fields) for case, fields in out.items()}
