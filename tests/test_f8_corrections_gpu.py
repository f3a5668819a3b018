"""GPU: the variant network's GEMMs with e4m3 correction products (tcgen05 kind::f16 main product and kind::f8f6f4 corrections
summed into one fp32 accumulator) against a float64 emulation of the same operand rounding, a structured product that is exact
only if every 8-bit tile and descriptor is laid out right, and the network with f8_mask 0 / 0x1f against the CPU oracle."""
import ctypes as C
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
TOL = 1e-3
MARGIN = 1e-4


def _gemm_f8(A, W, b, lo, f8):
    from pepper_b200 import _lib
    L = _lib.lib()
    L.pb_test_tc_gemm_f8.argtypes = [C.c_int] * 3 + [C.c_void_p] * 4 + [C.c_int, C.c_int]
    M, K = A.shape
    N = W.shape[0]
    out = np.zeros((M, N), np.float32)
    _lib.check(L.pb_test_tc_gemm_f8(M, N, K, A.ctypes.data, W.ctypes.data, b.ctypes.data, out.ctypes.data, lo, f8), "pb_test_tc_gemm_f8")
    return out


def _f16(x):
    return np.clip(x, -65504, 65504).astype(np.float16).astype(np.float64)


def _e4m3(x):
    return torch.from_numpy(np.clip(x, -448, 448).astype(np.float32)).to(torch.float8_e4m3fn).to(torch.float64).numpy()


def _emulate(A, W, b, lo, f8):
    """The operand images of tc_gemm.cuh ("e4m3 correction operands") and their products, accumulated in float64."""
    E = np.frexp(np.abs(W).max())[1]
    v = W.astype(np.float64) * 2.0 ** (12 - E)                    # exact: power-of-two scale of fp32 values
    w_hi = _f16(v)
    w_lo = v - w_hi
    a = A.astype(np.float64)
    a_hi = _f16(a)
    a_lo = a - a_hi
    if f8:
        acc = a_hi @ w_hi.T + _e4m3(a) @ _e4m3(w_lo).T
        if lo:
            acc += _e4m3(a_lo * 4096.0) @ _e4m3(v / 4096.0).T
    else:
        acc = a_hi @ w_hi.T + a_hi @ _f16(w_lo).T
        if lo:
            acc += _f16(a_lo) @ w_hi.T
    return acc * 2.0 ** (E - 12) + b


@pytest.mark.parametrize("M,N,K", [(128, 256, 32), (100, 256, 288), (300, 512, 768), (257, 256, 2048)])
@pytest.mark.parametrize("lo", [1, 0])
def test_f8_gemm_vs_emulation(M, N, K, lo):
    rng = np.random.default_rng(M + N + K + lo)
    A = rng.standard_normal((M, K)).astype(np.float32)
    W = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    b = rng.standard_normal(N).astype(np.float32)
    got = _gemm_f8(A, W, b, lo, 1)
    noise = 2e-6 * (np.abs(A).astype(np.float64) @ np.abs(W).T.astype(np.float64)).max()   # fp32 accumulation order
    err = np.abs(got - _emulate(A, W, b, lo, 1)).max()
    assert err < noise, (err, noise)
    exact = A.astype(np.float64) @ W.astype(np.float64).T + b
    assert np.abs(got - exact).max() < (2e-4 if lo else 2e-3)
    # the scaled fp16 images of the same weights (f8_mask bit clear)
    got16 = _gemm_f8(A, W, b, lo, 0)
    assert np.abs(got16 - _emulate(A, W, b, lo, 0)).max() < noise
    assert np.abs(got16 - exact).max() < (2e-4 if lo else 2e-3)


@pytest.mark.parametrize("M,N,K", [(128, 256, 32), (257, 512, 288)])
@pytest.mark.parametrize("lo", [1, 0])
def test_f8_gemm_structured(M, N, K, lo):
    """Every e4m3 product is exact and lands on one output column: a = k + j * 2^-13 (k in +-2..8, j in -3..3) and one-hot
    weights w = 0.5 + 2^-13 give a_hi = k (|j| 2^-13 is below half an fp16 ulp from 2 up), e4m3(a) = k, e4m3(a_lo * 2^12) = j / 2, fp16 w image 2048 + 0.5 and e4m3 images
    w_hi = 0.5, w_lo * 2^12 = 0.5, so out = (2048 k + k / 2 + lo * j / 4) / 4096 exactly — a misplaced 8-bit tile row, k chunk
    or descriptor moves the k / 2 or j / 4 term to another column."""
    rng = np.random.default_rng(M + K + lo)
    k = rng.integers(2, 9, size=(M, K)) * rng.choice([-1, 1], size=(M, K))
    j = rng.integers(-3, 4, size=(M, K))
    A = (k + j * 2.0 ** -13).astype(np.float32)
    cols = [(7 * n + 3) % K for n in range(N)]
    W = np.zeros((N, K), np.float32)
    W[np.arange(N), cols] = 0.5 + 2.0 ** -13
    zb = np.zeros(N, np.float32)
    got = _gemm_f8(A, W, zb, lo, 1)
    want = ((2048.0 + 0.5) * k[:, cols] + lo * 0.25 * j[:, cols]) / 4096.0
    assert np.array_equal(got, want.astype(np.float32)), np.abs(got - want).max()


@pytest.mark.parametrize("f8_mask", [0x1f, 0])
@pytest.mark.parametrize("n,seed", [(130, 2), (700, 3)])
def test_variant_net_f8_mask_vs_oracle(n, seed, f8_mask):
    from oracle import nets
    from pepper_b200.variant import VariantNet
    from tests.test_nets_gpu import _variant_images
    state = nets.make_variant_weights(seed)
    x = _variant_images(n, seed)
    want, whid = nets.variant_predict(state, x, threads=8, return_hidden=True)
    net = VariantNet(state)
    net.set_f8_mask(f8_mask)
    got, hid = net.predict(x, return_hidden=True)
    assert np.abs(hid - whid).max() < TOL, np.abs(hid - whid).max()
    assert np.abs(got - want).max() < TOL, np.abs(got - want).max()
    srt = np.sort(want, axis=1)
    clear = (srt[:, -1] - srt[:, -2]) > MARGIN
    assert np.array_equal(got.argmax(1)[clear], want.argmax(1)[clear])
    net.close()
