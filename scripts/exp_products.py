#!/usr/bin/env python
"""GPU experiment behind DESIGN.md's "two-product variant" table (VERDICT r1 item 2): for every choice of which GEMMs keep the
third tensor-core product (a_lo x w_hi), the measured error against the fp32 CPU oracle — max |dh| over all hidden states,
max |dp| / |dacc|, class indices that differ outside the 1e-4 margin — and the network time of a fixed batch.
    python scripts/exp_products.py > gpurun_out/r2_exp_products.json"""
import json
import os
import sys
import time
import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import nets  # noqa: E402  (a development script)
from pepper_b200.variant import VariantNet  # noqa: E402
from pepper_b200.polish import PolishNet  # noqa: E402
from pepper_b200 import weights  # noqa: E402
from tests.test_nets_gpu import _variant_images, _polish_images  # noqa: E402

out = {"variant": [], "polish": []}
if len(sys.argv) > 1 and sys.argv[1] == "f8":
    # `exp_products.py f8`: the variant net at the default lo_mask with each f8_mask choice — error against the oracle and the
    # device time of every kernel of one 9,472-candidate chunk (torch.profiler, in launch order)
    import torch
    F8 = {0x1f: "every correction in e4m3 (default)", 0x00: "fp16 split everywhere", 0x1e: "encoder fp16, rest e4m3",
          0x07: "LSTM layers e4m3, head fp16", 0x18: "head e4m3, LSTM layers fp16"}
    big = _variant_images(9472, 11)
    tnet = VariantNet(weights.random_variant_state(0))
    for mask, name in F8.items():
        row = {"f8_mask": mask, "what": name, "max_dh": 0.0, "max_dp": 0.0, "argmax_mismatch_outside_margin": 0, "n": 0}
        for seed in (1, 2, 3):
            state = nets.make_variant_weights(seed)
            x = _variant_images(700, seed)
            want, whid = nets.variant_predict(state, x, threads=16, return_hidden=True)
            net = VariantNet(state)
            net.set_f8_mask(mask)
            got, hid = net.predict(x, return_hidden=True)
            net.close()
            srt = np.sort(want, axis=1)
            clear = (srt[:, -1] - srt[:, -2]) > 1e-4
            row["max_dh"] = max(row["max_dh"], float(np.abs(hid - whid).max()))
            row["max_dp"] = max(row["max_dp"], float(np.abs(got - want).max()))
            row["argmax_mismatch_outside_margin"] += int((got.argmax(1)[clear] != want.argmax(1)[clear]).sum())
            row["n"] += int(clear.sum())
        tnet.set_f8_mask(mask)
        for _ in range(3):
            tnet.predict(big)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            tnet.predict(big)
        ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.name.startswith(("void pb::tc::k_", "pb::tc::k_"))),
                    key=lambda e: e.time_range.start)
        row["kernel_ms_one_chunk"] = [[e.name.split("(")[0].replace("void ", ""), round(e.device_time / 1e3, 3)] for e in ev]
        out["variant"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    tnet.close()
    print(json.dumps(out))
    sys.exit(0)
VN = {0x1f: "all x3", 0x1e: "encoder h x2", 0x1d: "decoder x x2", 0x1b: "decoder h x2", 0x17: "linear_1 x2", 0x0f: "linear_2-5 x2",
      0x1a: "encoder h + decoder h x2 (shipped default)", 0x18: "both LSTM layers x2, head x3", 0x07: "head x2, LSTM x3", 0x00: "all x2"}
if len(sys.argv) > 1:                       # e.g. `exp_products.py 0x1f,0x1a`: only these variant masks, polish skipped
    keep = {int(m, 0) for m in sys.argv[1].split(",")}
    VN = {m: n for m, n in VN.items() if m in keep}
big = _variant_images(9472 * 4, 11)
tnet = VariantNet(weights.random_variant_state(0))
for mask, name in VN.items():
    row = {"mask": mask, "what": name, "max_dh": 0.0, "max_dp": 0.0, "argmax_mismatch_outside_margin": 0, "n": 0}
    for seed in (1, 2, 3, 4, 5, 6) if len(sys.argv) > 1 else (1, 2, 3):
        state = nets.make_variant_weights(seed)
        x = _variant_images(700, seed)
        want, whid = nets.variant_predict(state, x, threads=16, return_hidden=True)
        net = VariantNet(state)
        net.set_lo_mask(mask)
        got, hid = net.predict(x, return_hidden=True)
        net.close()
        srt = np.sort(want, axis=1)
        clear = (srt[:, -1] - srt[:, -2]) > 1e-4
        row["max_dh"] = max(row["max_dh"], float(np.abs(hid - whid).max()))
        row["max_dp"] = max(row["max_dp"], float(np.abs(got - want).max()))
        row["argmax_mismatch_outside_margin"] += int((got.argmax(1)[clear] != want.argmax(1)[clear]).sum())
        row["n"] += int(clear.sum())
    tnet.set_lo_mask(mask)
    tnet.predict(big[:9472])
    ts = []
    for _ in range(3):
        t0 = time.perf_counter(); tnet.predict(big); ts.append(time.perf_counter() - t0)
    row["ms_per_37888_candidates_host_api"] = min(ts) * 1e3
    out["variant"].append(row)
    print(json.dumps(row), file=sys.stderr, flush=True)
tnet.close()
PN = {0x7: "all x3 (default)", 0x6: "encoder h x2", 0x5: "decoder x x2", 0x3: "decoder h x2", 0x0: "all x2"}
if len(sys.argv) > 1:
    PN = {}
bigp = _polish_images(1184, 12)
pnet = PolishNet(weights.random_polish_state(0))
for mask, name in PN.items():
    row = {"mask": mask, "what": name, "max_dh": 0.0, "max_dacc": 0.0, "argmax_mismatch_outside_margin": 0, "n": 0}
    for seed, n in ((4, 60), (6, 140)):
        state = nets.make_polish_weights(seed)
        x = _polish_images(n, seed)
        wb, wp, wh, wa = nets.polish_predict(state, x, threads=16)
        net = PolishNet(state)
        net.set_lo_mask(mask)
        bases, phred, hid, acc = net.predict(x, debug=True)
        net.close()
        srt = np.sort(wa, axis=2)
        clear = (srt[:, :, -1] - srt[:, :, -2]) > 1e-4
        row["max_dh"] = max(row["max_dh"], float(np.abs(hid - wh).max()))
        row["max_dacc"] = max(row["max_dacc"], float(np.abs(acc - wa).max()))
        row["argmax_mismatch_outside_margin"] += int((bases[clear] != wb[clear]).sum())
        row["n"] += int(clear.sum())
    pnet.set_lo_mask(mask)
    pnet.predict(bigp[:128])
    ts = []
    for _ in range(3):
        t0 = time.perf_counter(); pnet.predict(bigp); ts.append(time.perf_counter() - t0)
    row["ms_per_1184_images_host_api"] = min(ts) * 1e3
    out["polish"].append(row)
    print(json.dumps(row), file=sys.stderr, flush=True)
pnet.close()
print(json.dumps(out))
