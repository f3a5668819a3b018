"""CPU emulation of the tensor-core operand splits considered for the network kernels (round 2, VERDICT item 2).

Every GEMM of the two networks is re-evaluated with operands rounded the way a given scheme would feed them to
tcgen05.mma (fp32 accumulate; products of 16-bit operands are exact in fp32), and the hidden states / probabilities are
compared with the fp32 CPU oracle.  Used to choose the scheme before spending GPU time; the GPU tests are the gate.

    python scripts/sim_precision.py variant|polish [n] [scheme,scheme,...]

A scheme may name one choice per GEMM slot, separated by "/": variant slots are encoder, decoder x-part, decoder h-part,
linear_1, linear_2-5, so the shipped variant path is "f8w/f8b/f8w/f8b/f8b" (lo_mask 0x1a with every correction in e4m3;
the encoder's x-part is exact in fp16, so f8w and f8b agree there).
"""
import sys
import os
import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import nets  # noqa: E402  (a development script, not product code)

torch.set_num_threads(8)


def rn16(x, dt):
    return x.to(dt).to(torch.float64)


def e4m3(x):
    return x.clamp(-448.0, 448.0).to(torch.float8_e4m3fn).to(torch.float64)


def split(x, dt):
    hi = rn16(x, dt)
    lo = rn16(x - hi, dt)
    return hi, lo


class Scheme:
    """mm(a, W) with a [B,K] float64 activations, W [N,K] weights (fp32 values)."""

    def __init__(self, name):
        self.name = name
        self.cache = {}

    def wsplit(self, W, dt, scale=True):
        key = (id(W), dt)
        if key not in self.cache:
            W64 = W.to(torch.float64)
            s = 1.0
            if scale and dt == torch.float16:
                # per-tensor power-of-two scale so that max|w| lands in [2^-1, 1): keeps w_lo out of fp16 subnormals
                m = W64.abs().max().item()
                s = 2.0 ** (-np.ceil(np.log2(m))) if m > 0 else 1.0
            hi, lo = split(W64 * s, dt)
            self.cache[key] = (hi, lo, s)
        return self.cache[key]

    def mm(self, a, W, exact_a=False, slot=0):
        n = self.name
        if "/" in n:
            n = n.split("/")[slot]
        a = a.to(torch.float64)
        if n == "fp32":
            return (a.float() @ W.float().T).double()
        if n == "bf16x3":
            wh, wl, s = self.wsplit(W, torch.bfloat16)
            ah, al = split(a, torch.bfloat16)
            return ah @ wh.T + ah @ wl.T + al @ wh.T
        if n == "f16x3":
            wh, wl, s = self.wsplit(W, torch.float16)
            ah, al = split(a, torch.float16)
            return (ah @ wh.T + ah @ wl.T + al @ wh.T) / s
        if n == "f16x2":          # a_hi * (w_hi + w_lo)
            wh, wl, s = self.wsplit(W, torch.float16)
            ah = rn16(a, torch.float16)
            return (ah @ wh.T + ah @ wl.T) / s
        if n == "f16x2a":         # (a_hi + a_lo) * w_hi
            wh, wl, s = self.wsplit(W, torch.float16)
            ah, al = split(a, torch.float16)
            return (ah @ wh.T + al @ wh.T) / s
        if n == "f16x1":
            wh, wl, s = self.wsplit(W, torch.float16)
            ah = rn16(a, torch.float16)
            return (ah @ wh.T) / s
        if n == "bf16x2":
            wh, wl, s = self.wsplit(W, torch.bfloat16)
            ah = rn16(a, torch.bfloat16)
            return ah @ wh.T + ah @ wl.T
        if n in ("f8b", "f8w"):   # fp16 a_hi*w_hi + e4m3 corrections at a 2^12 scale (tc_gemm.cuh "e4m3 correction operands")
            wh, wl, s = self.wsplit(W, torch.float16)
            wl = W.to(torch.float64) * s - wh                      # exact residual: the e4m3 image rounds it once
            ah = rn16(a, torch.float16)
            out = ah @ wh.T + e4m3(a) @ e4m3(wl * 4096.0).T / 4096.0
            if n == "f8b":        # both corrections; f8w: a_hi*w_lo only
                out = out + e4m3((a - ah) * 4096.0) @ e4m3(wh).T / 4096.0
            return out / s
        raise ValueError(n)


def lstm_dir(S, x, Wih, Whh, b, reverse, slots=(0, 0)):
    B, T, _ = x.shape
    H = Whh.shape[1]
    h = torch.zeros(B, H, dtype=torch.float64)
    c = torch.zeros(B, H, dtype=torch.float64)
    out = torch.zeros(B, T, H, dtype=torch.float64)
    ts = range(T - 1, -1, -1) if reverse else range(T)
    for t in ts:
        g = S.mm(x[:, t], Wih, slot=slots[0]) + S.mm(h, Whh, slot=slots[1]) + b
        g = g.float()       # epilogue works in fp32
        i, f, gg, o = g.chunk(4, dim=1)
        c = (torch.sigmoid(f) * c.float() + torch.sigmoid(i) * torch.tanh(gg))
        h = (torch.sigmoid(o) * torch.tanh(c)).double()
        c = c.double()
        out[:, t] = h
    return out


def variant_forward(S, st, x):
    x = x.double()
    for layer in ("encoder", "decoder"):
        outs = []
        for suf, rev in (("", False), ("_reverse", True)):
            b = (st[f"{layer}.bias_ih_l0{suf}"] + st[f"{layer}.bias_hh_l0{suf}"]).double()
            outs.append(lstm_dir(S, x, st[f"{layer}.weight_ih_l0{suf}"], st[f"{layer}.weight_hh_l0{suf}"], b, rev,
                                 slots=(0, 0) if layer == "encoder" else (1, 2)))
        x = torch.cat(outs, dim=2)
    hid = x
    y = x.flatten(1, 2)
    for i in range(1, 6):
        y = torch.selu((S.mm(y, st[f"linear_{i}.weight"], slot=3 if i == 1 else 4) + st[f"linear_{i}.bias"].double()).float()).double()
    logits = y.float() @ st["output_layer_type.weight"].float().T + st["output_layer_type.bias"].float()
    return torch.softmax(logits, dim=1), hid


def gru_dir(S, x, h0, Wih, Whh, bih, bhh, reverse):
    B, T, _ = x.shape
    H = Whh.shape[1]
    h = h0.double()
    out = torch.zeros(B, T, H, dtype=torch.float64)
    ts = range(T - 1, -1, -1) if reverse else range(T)
    for t in ts:
        gi = (S.mm(x[:, t], Wih) + bih).float()
        gh = (S.mm(h, Whh) + bhh).float()
        ir, iz, in_ = gi.chunk(3, 1)
        hr, hz, hn = gh.chunk(3, 1)
        r = torch.sigmoid(ir + hr)
        z = torch.sigmoid(iz + hz)
        n = torch.tanh(in_ + r * hn)
        h = ((1 - z) * n + z * h.float()).double()
        out[:, t] = h
    return out, h


def polish_forward(S, st, images):
    B = images.shape[0]
    hidden = torch.zeros(B, 2, 128, dtype=torch.float64)
    acc = torch.zeros(B, 1000, 5)
    hids = []
    for i in range(0, 1000, 50):
        if i + 100 > 1000:
            break
        x = images[:, i:i + 100].double()
        hs = []
        outs = []
        for d, (suf, rev) in enumerate((("", False), ("_reverse", True))):
            o, h = gru_dir(S, x, hidden[:, d], st[f"gru_encoder.weight_ih_l0{suf}"], st[f"gru_encoder.weight_hh_l0{suf}"],
                           st[f"gru_encoder.bias_ih_l0{suf}"].double(), st[f"gru_encoder.bias_hh_l0{suf}"].double(), rev)
            outs.append(o); hs.append(h)
        x1 = torch.cat(outs, 2)
        outs2, hs2 = [], []
        for d, (suf, rev) in enumerate((("", False), ("_reverse", True))):
            o, h = gru_dir(S, x1, hs[d], st[f"gru_decoder.weight_ih_l0{suf}"], st[f"gru_decoder.weight_hh_l0{suf}"],
                           st[f"gru_decoder.bias_ih_l0{suf}"].double(), st[f"gru_decoder.bias_hh_l0{suf}"].double(), rev)
            outs2.append(o); hs2.append(h)
        y = torch.cat(outs2, 2).float()
        hidden = torch.stack(hs2, 1)
        hids.append(hidden.float().numpy())
        out = y @ st["dense1.weight"].float().T + st["dense1.bias"].float()
        acc[:, i:i + 100] += torch.softmax(out, 2)
    return acc.numpy(), np.stack(hids)


def main():
    which = sys.argv[1]
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 256
    schemes = sys.argv[3].split(",") if len(sys.argv) > 3 else ["bf16x3", "f16x3", "f16x2", "f16x2a", "f16x1", "bf16x2"]
    if which == "variant":
        for seed in (1, 2):
            st = nets.make_variant_weights(seed)
            rng = np.random.default_rng(seed)
            x = rng.integers(-40, 41, size=(n, 33, 26)).astype(np.int8)
            x[:, :, 0] = rng.integers(1, 6, size=(n, 33))
            x[rng.random((n, 33, 26)) < 0.5] = 0
            want, whid = nets.variant_predict(st, x, threads=8, return_hidden=True)
            for name in schemes:
                S = Scheme(name)
                p, hid = variant_forward(S, st, torch.from_numpy(x.astype(np.float32)))
                eh = np.abs(hid.numpy() - whid).max()
                ep = np.abs(p.numpy() - want).max()
                srt = np.sort(want, 1)
                clear = (srt[:, -1] - srt[:, -2]) > 1e-4
                am = (p.numpy().argmax(1)[clear] != want.argmax(1)[clear]).sum()
                print(f"variant seed {seed} {name:8s} max|dh| {eh:.2e}  max|dp| {ep:.2e}  argmax mismatches (clear) {am}", flush=True)
    else:
        for seed in (4, 6):
            st = nets.make_polish_weights(seed)
            rng = np.random.default_rng(seed)
            x = np.zeros((n, 1000, 10), np.uint8)
            cov = rng.integers(0, 255, size=(n, 1000, 1))
            x[:] = (rng.random((n, 1000, 10)) < 0.25) * cov
            wb, wp, wh, wa = nets.polish_predict(st, x, threads=8)
            for name in schemes:
                S = Scheme(name)
                acc, hid = polish_forward(S, st, torch.from_numpy(x.astype(np.float32)))
                eh = np.abs(hid - wh).max()
                ea = np.abs(acc - wa).max()
                srt = np.sort(wa, 2)
                clear = (srt[:, :, -1] - srt[:, :, -2]) > 1e-4
                am = (acc.argmax(2)[clear] != wa.argmax(2)[clear]).sum()
                print(f"polish seed {seed} {name:8s} max|dh| {eh:.2e}  max|dacc| {ea:.2e}  argmax mismatches (clear) {am}", flush=True)


if __name__ == "__main__":
    main()
