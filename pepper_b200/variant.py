"""Host side of the variant path: batched encoder + network wrappers over the C-ABI.

Mirrors the reference's operator surface for this path:

* ``VariantEncoder.encode`` == many ``RegionalSummaryGenerator(...).generate_summary(...)`` calls
  (pepper_variant/modules/python/AlignmentSummarizer.py:220-238) in one launch sequence;
* ``VariantNet.predict`` == ``TransducerGRU.forward`` as driven by
  pepper_variant/modules/python/models/predict_distributed_gpu.py:58-70.

The drop-in classes with the reference's own names live in ``pepper_b200/build/PEPPER_VARIANT.py``.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
import numpy as np

from . import _lib
from .abi import (HostReads, PbReads, PbRegion, PbVariantParams, regions_array, variant_params, WINDOW, FEATURES,
                  ALLELE_STRIDE, PB_ERR_CAPACITY)
from .synth import ReadBatch, RegionTable


@dataclass
class VariantCandidates:
    images: np.ndarray       # int8  [N,33,26]
    positions: np.ndarray    # int64 [N]
    depths: np.ndarray       # uint8 [N]
    freqs: np.ndarray        # uint8 [N]
    keys_raw: np.ndarray     # uint8 [N,64]
    region_of: np.ndarray    # int32 [N]
    n_per_region: np.ndarray  # int64 [n_regions]

    @property
    def keys(self) -> list[str]:
        return [bytes(k).split(b"\0", 1)[0].decode() for k in self.keys_raw]

    def __len__(self) -> int:
        return int(self.positions.shape[0])


def _bind(L):
    if getattr(L, "_variant_bound", False):
        return
    vp = C.c_void_p
    L.pb_variant_encoder_create.argtypes = [C.POINTER(vp), C.c_int]
    L.pb_variant_encoder_destroy.argtypes = [vp]
    L.pb_variant_encoder_set_debug.argtypes = [vp, C.c_int]
    L.pb_variant_encode_host.argtypes = [vp, C.POINTER(PbReads), C.POINTER(PbRegion), C.c_int64, vp, C.c_int64,
                                         C.POINTER(PbVariantParams), C.c_int64, vp, vp, vp, vp, vp, vp, vp,
                                         C.POINTER(C.c_int64), vp]
    L.pb_variant_encode_device.argtypes = [vp, C.POINTER(PbReads), vp, C.c_int64, C.POINTER(PbRegion), vp, C.c_int64,
                                           C.POINTER(PbVariantParams), C.c_int64, vp, vp, vp, vp, vp, vp, vp,
                                           C.POINTER(C.c_int64), vp]
    L.pb_variant_encoder_debug_region.argtypes = [vp, C.c_int64, vp, vp, vp, vp, vp]
    L.pb_variant_encoder_timings.argtypes = [vp, vp]
    L._variant_bound = True


class VariantEncoder:
    """Batched RegionalSummaryGenerator on one GPU."""

    def __init__(self, device: int = 0, debug: bool = False):
        _lib.require_gpu()
        self.L = _lib.lib()
        _bind(self.L)
        self.h = C.c_void_p()
        _lib.check(self.L.pb_variant_encoder_create(C.byref(self.h), device), "pb_variant_encoder_create")
        if debug:
            _lib.check(self.L.pb_variant_encoder_set_debug(self.h, 1), "set_debug")
        self.device = device

    def close(self):
        if self.h:
            self.L.pb_variant_encoder_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def encode(self, reads: ReadBatch, regions: RegionTable, params: dict, capacity: int | None = None,
               stream: int = 0) -> VariantCandidates:
        """Host buffers in, host buffers out (pb_variant_encode_host)."""
        hr = HostReads(reads)
        regs, keep = regions_array(regions)
        ref = np.ascontiguousarray(regions.ref, dtype=np.uint8)
        p = variant_params(**params)
        n_regions = regions.n_regions
        if capacity is None:
            span = int((regions.col("cand_end") - regions.col("cand_start") + 1).sum())
            capacity = max(1024, span // 16)
        while True:
            img = np.empty((capacity, WINDOW, FEATURES), dtype=np.int8)
            pos = np.empty(capacity, dtype=np.int64)
            dep = np.empty(capacity, dtype=np.uint8)
            frq = np.empty(capacity, dtype=np.uint8)
            keys = np.empty((capacity, ALLELE_STRIDE), dtype=np.uint8)
            rof = np.empty(capacity, dtype=np.int32)
            npr = np.zeros(max(n_regions, 1), dtype=np.int64)
            n = C.c_int64(0)
            rc = self.L.pb_variant_encode_host(self.h, C.byref(hr.struct), regs, n_regions, ref.ctypes.data,
                                               ref.shape[0], C.byref(p), capacity, img.ctypes.data, pos.ctypes.data,
                                               dep.ctypes.data, frq.ctypes.data, keys.ctypes.data, rof.ctypes.data,
                                               npr.ctypes.data, C.byref(n), C.c_void_p(stream))
            if rc == PB_ERR_CAPACITY:
                capacity = int(n.value) + 16
                continue
            _lib.check(rc, "pb_variant_encode_host")
            k = int(n.value)
            return VariantCandidates(img[:k], pos[:k], dep[:k], frq[:k], keys[:k], rof[:k], npr[:n_regions])

    def debug_region(self, region: int, L1: int):
        m = np.zeros((L1, FEATURES), dtype=np.int32)
        v = [np.zeros(L1, dtype=np.int32) for _ in range(4)]
        _lib.check(self.L.pb_variant_encoder_debug_region(self.h, region, m.ctypes.data, *[x.ctypes.data for x in v]),
                   "pb_variant_encoder_debug_region")
        return (m, *v)

    def timings(self) -> dict:
        ms = (C.c_float * 5)()
        _lib.check(self.L.pb_variant_encoder_timings(self.h, ms), "timings")
        return dict(zip(("prefix", "count", "sites", "alleles", "windows"), [float(x) for x in ms]))


def _state_arrays(L, state: dict, n_params: int, name_fn, numel_fn):
    """state_dict (torch tensors or numpy arrays, optionally with the DataParallel 'module.' prefix the reference
    strips in ModelHander.py:104-108) -> list of contiguous fp32 arrays in C-ABI order."""
    arrs = []
    for i in range(n_params):
        name = name_fn(i).decode()
        v = state.get(name, state.get("module." + name))
        if v is None:
            raise _lib.PepperB200Error(f"state_dict lacks parameter {name}")
        if hasattr(v, "detach"):
            v = v.detach().cpu().numpy()
        a = np.ascontiguousarray(v, dtype=np.float32)
        if a.size != numel_fn(i):
            raise _lib.PepperB200Error(f"parameter {name} has {a.size} elements, expected {numel_fn(i)}")
        arrs.append(a)
    return arrs


class VariantNet:
    """bi-LSTM x2 + MLP head on one GPU (pb_variant_net_*)."""

    def __init__(self, state: dict, device: int = 0):
        _lib.require_gpu()
        self.L = L = _lib.lib()
        vp = C.c_void_p
        L.pb_variant_net_param_name.restype = C.c_char_p
        L.pb_variant_net_param_name.argtypes = [C.c_int]
        L.pb_variant_net_param_numel.restype = C.c_int64
        L.pb_variant_net_param_numel.argtypes = [C.c_int]
        L.pb_variant_net_create.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(vp)]
        L.pb_variant_net_destroy.argtypes = [vp]
        L.pb_variant_net_forward_host.argtypes = [vp, vp, C.c_int64, vp, vp, vp]
        L.pb_variant_net_forward_device.argtypes = [vp, vp, C.c_int64, vp, vp, vp]
        L.pb_variant_net_launches.argtypes = [vp, C.POINTER(C.c_int64)]
        L.pb_variant_net_set_mode.argtypes = [vp, C.c_int]
        n = 28
        arrs = _state_arrays(L, state, n, L.pb_variant_net_param_name, L.pb_variant_net_param_numel)
        ptrs = (vp * n)(*[a.ctypes.data for a in arrs])
        self.h = vp()
        _lib.check(L.pb_variant_net_create(C.byref(self.h), device, ptrs), "pb_variant_net_create")

    def close(self):
        if self.h:
            self.L.pb_variant_net_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def predict(self, images_i8: np.ndarray, return_hidden: bool = False, stream: int = 0):
        """int8 [N,33,26] host -> float32 probs [N,3] host (== predict_distributed_gpu.py:58-70)."""
        x = np.ascontiguousarray(images_i8, dtype=np.int8)
        n = x.shape[0]
        probs = np.empty((n, 3), dtype=np.float32)
        hid = np.empty((n, WINDOW, 512), dtype=np.float32) if return_hidden else None
        _lib.check(self.L.pb_variant_net_forward_host(self.h, x.ctypes.data, n, probs.ctypes.data,
                                                     hid.ctypes.data if return_hidden else None, C.c_void_p(stream)),
                   "pb_variant_net_forward_host")
        return (probs, hid) if return_hidden else probs

    def set_mode(self, mode: int) -> None:
        """0 = fp32 FFMA GEMMs, 1 = tcgen05 GEMMs with the 16-bit hi/lo operand split (2-3 products per GEMM, set_lo_mask; default)."""
        _lib.check(self.L.pb_variant_net_set_mode(self.h, mode), "pb_variant_net_set_mode")

    def set_lo_mask(self, mask: int) -> None:
        """Bit set = that GEMM keeps its third tensor-core product (a_lo x w_hi).  bits: 0 encoder h-part, 1 decoder x-part,
        2 decoder h-part, 3 linear_1, 4 linear_2-5.  Default 0x1a: the recurrent GEMMs pass the parity gate with two products
        (DESIGN.md section 4); 0x1f = three everywhere."""
        self.L.pb_variant_net_set_lo_mask.argtypes = [C.c_void_p, C.c_int]
        _lib.check(self.L.pb_variant_net_set_lo_mask(self.h, mask), "pb_variant_net_set_lo_mask")

    def set_f8_mask(self, mask: int) -> None:
        """Bit set (same bits as set_lo_mask) = that GEMM runs its correction products (a_hi x w_lo, and a_lo x w_hi where the
        lo mask keeps it) as e4m3 tensor-core MMAs next to the fp16 a_hi x w_hi.  Default 0x1f; 0 = the fp16 split everywhere."""
        self.L.pb_variant_net_set_f8_mask.argtypes = [C.c_void_p, C.c_int]
        _lib.check(self.L.pb_variant_net_set_f8_mask(self.h, mask), "pb_variant_net_set_f8_mask")

    def launches(self) -> int:
        n = C.c_int64(0)
        _lib.check(self.L.pb_variant_net_launches(self.h, C.byref(n)), "launches")
        return int(n.value)
