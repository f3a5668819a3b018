// Host side of the tcgen05 network path (mode 1): weight / operand tiling, per-layer launch sequences, and a
// GEMM self-test entry point.  Device code: tc_gemm.cuh.
#include "handles.cuh"
#include "tc_gemm.cuh"
#include <vector>
#include <algorithm>
#include <stdlib.h>

using namespace pb;
using tc::Args;
using tc::Dir;
using tc::Seg;
using tc::TILE_ELEMS;
typedef pb::tc::op_t bf16;      // 16-bit operand element (fp16 by default, bf16 with -DPB_OPERAND_BF16)

namespace pb {

static inline uint16_t f2bf(float f) { return tc::op_bits(f); }      // round to nearest even into the operand type
static inline float bf2f(uint16_t h) { return tc::op_val(h); }

// row-major [rows][K] fp32 (rows % 128 == 0 after padding, K % 32 == 0 after padding) -> hi / lo tiles [rt][kt][4][128][8] of
// v = src * scale.  With F8 set, also the e4m3 tiles [rt][kt][2][128][16]: hi8 = e4m3(v * F8->hi_scale), lo8 = e4m3((v - v_hi) *
// F8->lo_scale) — (2^-12, 1) for weights, (1, 2^12) for activations (tc_gemm.cuh, "e4m3 correction operands").
struct F8Tiles {
    std::vector<uint8_t> hi, lo;
    float hi_scale, lo_scale;
};
static void tile_matrix(const float *src, int64_t rows, int64_t K, int64_t rows_p, int64_t Kp, std::vector<uint16_t> &hi, std::vector<uint16_t> &lo,
                        int64_t TR = 128 /* rows per tile: 128 for A operands, 256 for the weights of the persistent kernel */,
                        float scale = 1.f, F8Tiles *F8 = nullptr) {
    const int64_t RT = rows_p / TR, KT = Kp / 32;
    hi.assign((size_t) (RT * KT * TR * 32), 0);
    lo.assign((size_t) (RT * KT * TR * 32), 0);
    if (F8) {
        F8->hi.assign(hi.size(), 0);
        F8->lo.assign(hi.size(), 0);
    }
    for (int64_t r = 0; r < rows; r++)
        for (int64_t k = 0; k < K; k++) {
            const float v = src[r * K + k] * scale;
            const uint16_t h = f2bf(v);
            const float res = v - bf2f(h);
            const int64_t tile = ((r / TR) * KT + k / 32) * (TR * 32);
            const int64_t o = tile + ((k % 32) / 8) * (TR * 8) + (r % TR) * 8 + (k % 8);
            hi[(size_t) o] = h;
            lo[(size_t) o] = f2bf(res);
            if (F8) {
                const int64_t o8 = tile + ((k % 32) / 16) * (TR * 16) + (r % TR) * 16 + (k % 16);
                F8->hi[(size_t) o8] = tc::f8_bits(v * F8->hi_scale);
                F8->lo[(size_t) o8] = tc::f8_bits(res * F8->lo_scale);
            }
        }
}

static int upload_tiles(DevBuf &dhi, DevBuf &dlo, const std::vector<uint16_t> &hi, const std::vector<uint16_t> &lo) {
    PB_TRY(dhi.reserve(hi.size() * 2));
    PB_TRY(dlo.reserve(lo.size() * 2));
    PB_CUDA(cudaMemcpy(dhi.p, hi.data(), hi.size() * 2, cudaMemcpyHostToDevice));
    PB_CUDA(cudaMemcpy(dlo.p, lo.data(), lo.size() * 2, cudaMemcpyHostToDevice));
    return PB_OK;
}
static int upload_f8(DevBuf &dhi, DevBuf &dlo, const F8Tiles &F) {
    PB_TRY(dhi.reserve(F.hi.size()));
    PB_TRY(dlo.reserve(F.lo.size()));
    PB_CUDA(cudaMemcpy(dhi.p, F.hi.data(), F.hi.size(), cudaMemcpyHostToDevice));
    PB_CUDA(cudaMemcpy(dlo.p, F.lo.data(), F.lo.size(), cudaMemcpyHostToDevice));
    return PB_OK;
}

// Weight images, optionally with the e4m3 correction images: the fp16 images then hold w * 2^(12-E), max|w * 2^-E| in
// [0.5, 1), and *acc_scale = 2^(E-12) maps the accumulator back.
static int upload_weight(const float *w, int64_t N, int64_t K, int64_t Np, int64_t Kp, bool with_f8, DevBuf &w_hi, DevBuf &w_lo, DevBuf &w8_hi,
                         DevBuf &w8_lo, float &acc_scale) {
    std::vector<uint16_t> hi, lo;
    if (!with_f8) {
        tile_matrix(w, N, K, Np, Kp, hi, lo, 256);
        acc_scale = 1.f;
        return upload_tiles(w_hi, w_lo, hi, lo);
    }
    float m = 0.f;
    for (int64_t i = 0; i < N * K; i++) m = std::max(m, fabsf(w[i]));
    int E = 0;
    if (m > 0.f) frexpf(m, &E);                              // m = f * 2^E, f in [0.5, 1)
    F8Tiles F{{}, {}, 1.f / tc::F8_LO_SCALE, 1.f};
    tile_matrix(w, N, K, Np, Kp, hi, lo, 256, ldexpf(1.f, 12 - E), &F);
    acc_scale = ldexpf(1.f, E - 12);
    PB_TRY(upload_tiles(w_hi, w_lo, hi, lo));
    return upload_f8(w8_hi, w8_lo, F);
}

// weights of one RNN direction, packed rows 4j+g (host copy kept by nets.cu) with K = [x | pad32 | h]
int tc_upload_rnn(TcRnn &T, const float *Wp /* [4H][Kp_src] */, int K0, int K0p_src, int H, int Kp_src, bool with_f8) {
    const int K0p = (K0 + 31) / 32 * 32;
    const int Kp = K0p + H;
    std::vector<float> W((size_t) 4 * H * Kp, 0.f);
    for (int n = 0; n < 4 * H; n++) {
        for (int k = 0; k < K0; k++) W[(size_t) n * Kp + k] = Wp[(size_t) n * Kp_src + k];
        for (int k = 0; k < H; k++) W[(size_t) n * Kp + K0p + k] = Wp[(size_t) n * Kp_src + K0p_src + k];
    }
    T.nkt_x = K0p / 32; T.nkt_h = H / 32;
    return upload_weight(W.data(), 4 * H, Kp, 4 * H, Kp, with_f8, T.w_hi, T.w_lo, T.w8_hi, T.w8_lo, T.acc_scale);
}
int tc_upload_lin(TcLin &T, const float *w, int N, int K, bool with_f8) {
    const int Np = (N + 255) / 256 * 256, Kp = (K + 31) / 32 * 32;
    T.nkt = Kp / 32;
    return upload_weight(w, N, K, Np, Kp, with_f8, T.w_hi, T.w_lo, T.w8_hi, T.w8_lo, T.acc_scale);
}

static int g_num_sms = 0;

// persistent 128x256-tile kernel (weights packed in 256-row tiles); `nt128` = number of 128-column tiles = N / 128
template <int EPI>
static int launch_tc(const Args &A, int mt, int nt128, int ndir, cudaStream_t st) {
    static bool attr_set = false;
    if (!attr_set) {
        PB_CUDA(cudaFuncSetAttribute(tc::k_tc_gemm_p<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::PSMEM_BYTES));
        attr_set = true;
    }
    if (g_num_sms == 0) {
        int dev = 0;
        PB_CUDA(cudaGetDevice(&dev));
        PB_CUDA(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
    }
    if (nt128 % 2) { set_error("tcgen05 path needs N %% 256 == 0"); return PB_ERR_ARG; }
    const int nt = nt128 / 2;
    const int tiles = mt * nt * ndir;
    tc::k_tc_gemm_p<EPI><<<(unsigned) std::min(tiles, g_num_sms), tc::PG_THREADS, tc::PSMEM_BYTES, st>>>(A, mt, nt, ndir);
    return PB_OK;
}
static Dir empty_dir() {
    Dir D;
    memset(&D, 0, sizeof(D));
    D.acc_scale = 1.f;
    return D;
}

// ------------------------------------------------------------------------------------------------- variant
constexpr int VT = 33, VH = 256;

// GEMM slots of lo_mask / f8_mask: 0 encoder (x- and h-part), 1 decoder x-part, 2 decoder h-part, 3 linear_1, 4 linear_2-5.
// An operand is written in the images its consumer GEMMs (slot bits `consumers`) read: fp16 hi always, fp16 lo where an fp16
// GEMM runs a_lo*w_hi, e4m3 hi where a GEMM runs its corrections in e4m3, e4m3 lo where such a GEMM also runs a_lo*w_hi.
struct OpImages { bool lo16, hi8, lo8; };
static OpImages op_images(const TcVariant &T, int consumers) {
    OpImages r{false, false, false};
    for (int i = 0; i < 5; i++) {
        if (!((consumers >> i) & 1)) continue;
        const bool lo = (T.lo_mask >> i) & 1, f8 = (T.f8_mask >> i) & 1;
        r.lo16 |= lo && !f8;
        r.hi8 |= f8;
        r.lo8 |= lo && f8;
    }
    return r;
}

int variant_forward_tc(pb_variant_net *N, const int8_t *d_images, int64_t B, float *d_probs, float *d_hidden_dbg, cudaStream_t st,
                       void (*out_kernel)(const float *, const float *, const float *, float *, int64_t, const OutSink &, cudaStream_t),
                       const OutSink &sink) {
    TcVariant &T = *N->tc;
    const int64_t Mt = ceil_div(B, 128), Bp = Mt * 128;
    const int64_t seq_tiles = Mt * VT * 16;                 // [mt][t][16 k-tiles] of a 512-feature sequence operand
    const size_t seq_bytes = (size_t) (seq_tiles * TILE_ELEMS) * 2, act_bytes = (size_t) (Mt * 16 * TILE_ELEMS) * 2;
    const OpImages enc_out = op_images(T, 0x3), dec_out = op_images(T, 0xc), act_out = op_images(T, 0x10);
    PB_TRY(T.img_op.reserve((size_t) (Mt * VT * TILE_ELEMS) * 2));
    PB_TRY(T.img_op8.reserve((size_t) (Mt * VT * TILE_ELEMS)));
    PB_TRY(T.yenc_hi.reserve(seq_bytes));
    PB_TRY(T.ydec_hi.reserve(seq_bytes));
    if (enc_out.lo16) PB_TRY(T.yenc_lo.reserve(seq_bytes));
    if (dec_out.lo16) PB_TRY(T.ydec_lo.reserve(seq_bytes));
    if (enc_out.hi8) PB_TRY(T.yenc_hi8.reserve(seq_bytes / 2));
    if (enc_out.lo8) PB_TRY(T.yenc_lo8.reserve(seq_bytes / 2));
    if (dec_out.hi8) PB_TRY(T.ydec_hi8.reserve(seq_bytes / 2));
    if (dec_out.lo8) PB_TRY(T.ydec_lo8.reserve(seq_bytes / 2));
    PB_TRY(T.c.reserve(sizeof(float) * 2 * VH * Bp));
    for (int i = 0; i < 2; i++) {
        PB_TRY(T.act_hi[i].reserve(act_bytes));
        if (act_out.lo16) PB_TRY(T.act_lo[i].reserve(act_bytes));
        if (act_out.hi8) PB_TRY(T.act_hi8[i].reserve(act_bytes / 2));
        if (act_out.lo8) PB_TRY(T.act_lo8[i].reserve(act_bytes / 2));
    }
    PB_TRY(T.final_f32.reserve(sizeof(float) * Bp * 512));
    auto pick16 = [](bool want, DevBuf &b) { return want ? b.as<bf16>() : nullptr; };
    auto pick8 = [](bool want, DevBuf &b) { return want ? b.as<uint8_t>() : nullptr; };
    const bool img8 = (T.f8_mask & 1) != 0;                 // the encoder's x-part reads e4m3 images

    tc::k_tc_pack_images<<<(unsigned) ceil_div(Bp * VT * 4, 256), 256, 0, st>>>(d_images, T.img_op.as<bf16>(), pick8(img8, T.img_op8), B, VT, 26);
    N->launches++;

    // A-operand segment at tile offset `off` of a sequence / activation operand, for a GEMM with the given lo / f8 bits
    auto seg = [](const bf16 *hi, const bf16 *lo16, const uint8_t *hi8, const uint8_t *lo8, int64_t off, int lo, int f8) {
        Seg S;
        memset(&S, 0, sizeof(S));
        S.hi = hi + off;
        if (f8) { S.hi8 = hi8 + off; S.lo8 = lo ? lo8 + off : nullptr; }
        else S.lo = lo ? lo16 + off : nullptr;
        return S;
    };
    for (int layer = 0; layer < 2; layer++) {
        PB_CUDA(cudaMemsetAsync(T.c.p, 0, sizeof(float) * 2 * VH * Bp, st));
        const OpImages &yo = layer == 0 ? enc_out : dec_out;
        bf16 *y_hi = layer == 0 ? T.yenc_hi.as<bf16>() : T.ydec_hi.as<bf16>();
        bf16 *y_lo = pick16(yo.lo16, layer == 0 ? T.yenc_lo : T.ydec_lo);
        uint8_t *y_hi8 = pick8(yo.hi8, layer == 0 ? T.yenc_hi8 : T.ydec_hi8), *y_lo8 = pick8(yo.lo8, layer == 0 ? T.yenc_lo8 : T.ydec_lo8);
        // slot bits of this layer's x-part and h-part
        const int sx = layer == 0 ? 0 : 1, sh = layer == 0 ? 0 : 2;
        const int lo_x = layer == 0 ? 0 : (T.lo_mask >> sx) & 1;        // encoder x-part: int8 images are exact (no lo operand at all)
        const int lo_h = (T.lo_mask >> sh) & 1, f8_x = (T.f8_mask >> sx) & 1, f8_h = (T.f8_mask >> sh) & 1;
        static const bool persist = !(getenv("PB_LSTM_PERSIST") && atoi(getenv("PB_LSTM_PERSIST")) == 0);
        if (persist) {
            // one launch per layer: every CTA keeps its (direction, row tile) for all 33 steps (k_lstm_layer)
            tc::LstmLayer L;
            memset(&L, 0, sizeof(L));
            if (layer == 0) {
                L.x_hi = T.img_op.as<bf16>(); L.x_hi8 = T.img_op8.as<uint8_t>();
                L.x_mt_stride = (int64_t) VT * TILE_ELEMS; L.x_nkt = 1;
            } else {
                L.x_hi = T.yenc_hi.as<bf16>(); L.x_lo = T.yenc_lo.as<bf16>(); L.x_hi8 = T.yenc_hi8.as<uint8_t>(); L.x_lo8 = T.yenc_lo8.as<uint8_t>();
                L.x_mt_stride = (int64_t) VT * 16 * TILE_ELEMS; L.x_nkt = 16;
            }
            for (int d = 0; d < 2; d++) {
                TcRnn &W = layer == 0 ? T.enc[d] : T.dec[d];
                L.w_hi[d] = W.w_hi.as<bf16>(); L.w_lo[d] = W.w_lo.as<bf16>();
                L.w8_hi[d] = W.w8_hi.as<uint8_t>(); L.w8_lo[d] = W.w8_lo.as<uint8_t>(); L.acc_scale[d] = W.acc_scale;
                L.bias[d] = (layer == 0 ? N->enc[d] : N->dec[d]).bias.as<float>();
                L.c[d] = T.c.as<float>() + (int64_t) d * VH * Bp;
                if (W.nkt_x != L.x_nkt || W.nkt_h != 8) { set_error("unexpected packed LSTM weight shape"); return PB_ERR_STATE; }
            }
            L.y_hi = y_hi; L.y_lo = y_lo; L.y_hi8 = y_hi8; L.y_lo8 = y_lo8; L.y_mt_stride = (int64_t) VT * 16 * TILE_ELEMS;
            if (layer == 1 && d_hidden_dbg) { L.y_f32 = d_hidden_dbg; L.ldy = (int64_t) VT * 512; }
            L.M = (int) B; L.n_mt = (int) Mt; L.T = VT; L.c_ld = Bp;
            L.lo_x = lo_x; L.lo_h = lo_h; L.f8_x = f8_x; L.f8_h = f8_h;
            static bool attr_set = false;
            if (!attr_set) {
                PB_CUDA(cudaFuncSetAttribute(tc::k_lstm_layer, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::PSMEM_BYTES));
                attr_set = true;
            }
            tc::k_lstm_layer<<<(unsigned) (2 * Mt), tc::PG_THREADS, tc::PSMEM_BYTES, st>>>(L);
            N->launches++;
            continue;
        }
        for (int t = 0; t < VT; t++) {
            Args A;
            A.M = (int) B; A.N = 4 * VH; A.c_ld = Bp;
            for (int d = 0; d < 2; d++) {
                const int tt = d == 0 ? t : VT - 1 - t;
                const int tp = d == 0 ? tt - 1 : tt + 1;
                Dir D = empty_dir();
                TcRnn &W = layer == 0 ? T.enc[d] : T.dec[d];
                if (layer == 0) {
                    D.seg[0] = seg(T.img_op.as<bf16>(), nullptr, T.img_op8.as<uint8_t>(), nullptr, (int64_t) tt * TILE_ELEMS, 0, f8_x);
                    D.seg[0].mt_stride = (int64_t) VT * TILE_ELEMS; D.seg[0].nkt = 1;
                } else {
                    D.seg[0] = seg(T.yenc_hi.as<bf16>(), T.yenc_lo.as<bf16>(), T.yenc_hi8.as<uint8_t>(), T.yenc_lo8.as<uint8_t>(),
                                   (int64_t) tt * 16 * TILE_ELEMS, lo_x, f8_x);
                    D.seg[0].mt_stride = (int64_t) VT * 16 * TILE_ELEMS; D.seg[0].nkt = 16;
                }
                if (t > 0) {
                    D.seg[1] = seg(y_hi, y_lo, y_hi8, y_lo8, ((int64_t) tp * 16 + d * 8) * TILE_ELEMS, lo_h, f8_h);
                    D.seg[1].mt_stride = (int64_t) VT * 16 * TILE_ELEMS; D.seg[1].nkt = 8;
                }
                D.w_hi = W.w_hi.as<bf16>(); D.w_lo = W.w_lo.as<bf16>(); D.w_nkt = W.nkt_x + W.nkt_h;
                D.w8_hi = W.w8_hi.as<uint8_t>(); D.w8_lo = W.w8_lo.as<uint8_t>(); D.acc_scale = W.acc_scale;
                D.bias = (layer == 0 ? N->enc[d] : N->dec[d]).bias.as<float>();
                D.c = T.c.as<float>() + (int64_t) d * VH * Bp;
                D.y_hi = y_hi; D.y_lo = y_lo; D.y_hi8 = y_hi8; D.y_lo8 = y_lo8;
                D.y_mt_stride = (int64_t) VT * 16 * TILE_ELEMS; D.y_kt0 = tt * 16 + d * 8;
                if (layer == 1 && d_hidden_dbg) { D.y_f32 = d_hidden_dbg + (int64_t) tt * 512 + d * VH; D.ldy = (int64_t) VT * 512; }
                A.d[d] = D;
            }
            PB_TRY(launch_tc<tc::EPI_LSTM>(A, (int) Mt, 4 * VH / 128, 2, st));
            N->launches++;
        }
    }
    // MLP head
    for (int i = 0; i < 5; i++) {
        Args A;
        A.M = (int) B; A.N = 512; A.c_ld = 0;
        Dir D = empty_dir();
        const int slot = i == 0 ? 3 : 4, lo = (T.lo_mask >> slot) & 1, f8 = (T.f8_mask >> slot) & 1;
        if (i == 0) {
            D.seg[0] = seg(T.ydec_hi.as<bf16>(), T.ydec_lo.as<bf16>(), T.ydec_hi8.as<uint8_t>(), T.ydec_lo8.as<uint8_t>(), 0, lo, f8);
            D.seg[0].mt_stride = (int64_t) VT * 16 * TILE_ELEMS; D.seg[0].nkt = VT * 16;
        } else {
            const int a = (i - 1) & 1;
            D.seg[0] = seg(T.act_hi[a].as<bf16>(), T.act_lo[a].as<bf16>(), T.act_hi8[a].as<uint8_t>(), T.act_lo8[a].as<uint8_t>(), 0, lo, f8);
            D.seg[0].mt_stride = (int64_t) 16 * TILE_ELEMS; D.seg[0].nkt = 16;
        }
        D.w_hi = T.lin[i].w_hi.as<bf16>(); D.w_lo = T.lin[i].w_lo.as<bf16>(); D.w_nkt = T.lin[i].nkt;
        D.w8_hi = T.lin[i].w8_hi.as<uint8_t>(); D.w8_lo = T.lin[i].w8_lo.as<uint8_t>(); D.acc_scale = T.lin[i].acc_scale;
        D.bias = N->lin[i].bias.as<float>();
        if (i < 4) {             // linear_5 feeds only the fp32 copy read by the output layer
            D.y_hi = T.act_hi[i & 1].as<bf16>(); D.y_lo = pick16(act_out.lo16, T.act_lo[i & 1]);
            D.y_hi8 = pick8(act_out.hi8, T.act_hi8[i & 1]); D.y_lo8 = pick8(act_out.lo8, T.act_lo8[i & 1]);
            D.y_mt_stride = (int64_t) 16 * TILE_ELEMS; D.y_kt0 = 0;
        } else {
            D.y_f32 = T.final_f32.as<float>(); D.ldy = 512;
        }
        A.d[0] = D; A.d[1] = D;
        PB_TRY(launch_tc<tc::EPI_SELU>(A, (int) Mt, 4, 1, st));
        N->launches++;
    }
    out_kernel(T.final_f32.as<float>(), N->outl.W.as<float>(), N->outl.bias.as<float>(), d_probs, B, sink, st);
    N->launches++;
    PB_CUDA(cudaGetLastError());
    return PB_OK;
}

// ------------------------------------------------------------------------------------------------- polish
constexpr int PH = 128, PWIN = 100;

// uint8 image window -> tiled operand [mt][100][1 k-tile] (values <= 254 are exact in bf16)
__global__ void k_tc_pack_polish(const uint8_t *__restrict__ img /* [B][1000][10] */, bf16 *__restrict__ op, int64_t B, int win_start) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;     // (row, t, kc)
    const int64_t total = ceil_div(B, 128) * 128 * PWIN * 4;
    if (i >= total) return;
    const int kc = (int) (i & 3);
    const int64_t rt = i >> 2;
    const int t = (int) (rt % PWIN);
    const int64_t row = rt / PWIN;
    uint32_t w[4] = {0, 0, 0, 0};
    if (row < B) {
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const int k = kc * 8 + e;
            const float v = (k < 10) ? (float) img[(row * 1000 + win_start + t) * 10 + k] : 0.f;
            w[e >> 1] |= (uint32_t) tc::op_bits(v) << (16 * (e & 1));
        }
    }
    const int64_t o = ((row >> 7) * PWIN + t) * TILE_ELEMS + kc * 1024 + (row & 127) * 8;
    *reinterpret_cast<uint4 *>(op + o) = make_uint4(w[0], w[1], w[2], w[3]);
}

// hidden state [B][2][128] fp32 out of a sequence operand (fwd: time 99, bwd: time 0), for the debug read-back
__global__ void k_tc_unpack_hidden(const bf16 *__restrict__ y_hi, const bf16 *__restrict__ y_lo, float *__restrict__ out, int64_t B) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * 2 * PH) return;
    const int j = (int) (i % PH);
    const int d = (int) ((i / PH) % 2);
    const int64_t b = i / (2 * PH);
    const int tt = d == 0 ? PWIN - 1 : 0;
    const int64_t o = (((b >> 7) * PWIN + tt) * 8 + d * 4 + (j >> 5)) * TILE_ELEMS + ((j & 31) >> 3) * 1024 + (b & 127) * 8 + (j & 7);
    out[i] = tc::op_val(reinterpret_cast<const uint16_t *>(y_hi)[o]) + tc::op_val(reinterpret_cast<const uint16_t *>(y_lo)[o]);
}
// dense1 (256 -> 5) + softmax + window accumulate straight from the decoder's tiled output operand
// (predict_distributed_cpu.py:62-81): one thread per (image row, time step); lanes = consecutive rows of a row tile, so
// every 16-byte operand load is coalesced; no fp32 copy of the decoder output is ever written.
__global__ void __launch_bounds__(128) k_polish_dense_tiles(const bf16 *__restrict__ y_hi, const bf16 *__restrict__ y_lo,
                                                            const float *__restrict__ W /* [5][256] */, const float *__restrict__ bias,
                                                            float *__restrict__ acc /* [B][1000][5] */, int64_t B, int win_start) {
    __shared__ float sW[5 * 256];
    for (int i = threadIdx.x; i < 5 * 256; i += 128) sW[i] = W[i];
    __syncthreads();
    const int64_t mt = blockIdx.x / PWIN;
    const int t = (int) (blockIdx.x % PWIN);
    const int r128 = threadIdx.x;
    const int64_t row = mt * 128 + r128;
    if (row >= B) return;
    float s[5] = {bias[0], bias[1], bias[2], bias[3], bias[4]};
    const int64_t tile0 = (mt * PWIN + t) * 8;
#pragma unroll 2
    for (int kt = 0; kt < 8; kt++) {
#pragma unroll
        for (int kc = 0; kc < 4; kc++) {
            const int64_t o = (tile0 + kt) * TILE_ELEMS + kc * 1024 + r128 * 8;
            const uint4 h = *reinterpret_cast<const uint4 *>(y_hi + o), l = *reinterpret_cast<const uint4 *>(y_lo + o);
            const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
            for (int e = 0; e < 8; e++) {
                const float v = tc::op_val(hw[e >> 1] >> (16 * (e & 1))) + tc::op_val(lw[e >> 1] >> (16 * (e & 1)));
                const int f = kt * 32 + kc * 8 + e;
#pragma unroll
                for (int c = 0; c < 5; c++) s[c] = fmaf(v, sW[c * 256 + f], s[c]);
            }
        }
    }
    float m = s[0];
#pragma unroll
    for (int c = 1; c < 5; c++) m = fmaxf(m, s[c]);
    float e[5], sum = 0.f;
#pragma unroll
    for (int c = 0; c < 5; c++) { e[c] = expf(s[c] - m); sum += e[c]; }
    float *dst = acc + (row * 1000 + win_start + t) * 5;
#pragma unroll
    for (int c = 0; c < 5; c++) dst[c] += e[c] / sum;
}

// one bidirectional GRU layer over the 100 steps of a window: ONE launch of k_gru_layer (or the k_gru_cluster fallback).
//   x operand: [mt][100][xkt] tiles (hi, lo or hi only); h0: the fwd state at time 99 / bwd state at time 0 of another
//   sequence operand (h0_is_seq) or the zero operand.
static int gru_layer_tc(pb_polish_net *N, TcRnn *W, DevRnn *Wb, const bf16 *x_hi, const bf16 *x_lo, int xkt, const bf16 *h0_hi,
                        const bf16 *h0_lo, bool h0_is_seq, bf16 *y_hi, bf16 *y_lo, int64_t B, cudaStream_t st) {
    static bool attr_set = false;
    if (!attr_set) {
        PB_CUDA(cudaFuncSetAttribute(tc::k_gru_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::CSMEM_BYTES));
        attr_set = true;
    }
    TcPolish &T = *N->tc;
    const int64_t Mt = ceil_div(B, 128);
    const int64_t ystride = (int64_t) PWIN * 8 * TILE_ELEMS;
    tc::GruWin G;
    G.x_hi = x_hi; G.x_lo = x_lo; G.x_kt = xkt;
    for (int d = 0; d < 2; d++) {
        const int t0 = d == 0 ? PWIN - 1 : 0;
        G.h0_hi[d] = h0_is_seq ? h0_hi + ((int64_t) t0 * 8 + d * 4) * TILE_ELEMS : h0_hi;
        G.h0_lo[d] = h0_is_seq ? h0_lo + ((int64_t) t0 * 8 + d * 4) * TILE_ELEMS : h0_lo;
        G.w_hi[d] = W[d].w_hi.as<bf16>(); G.w_lo[d] = W[d].w_lo.as<bf16>();
        G.bias[d] = Wb[d].bias.as<float>();
    }
    G.h0_mt_stride = h0_is_seq ? ystride : 0;
    G.y_hi = y_hi; G.y_lo = y_lo; G.flags = nullptr;
    G.M = (int) B; G.n_mt = (int) Mt; G.T = PWIN;
    G.lo_x = xkt == 1 ? 1 : ((T.lo_mask >> 1) & 1);                  // encoder x-part: uint8 images are exact
    G.lo_h = xkt == 1 ? (T.lo_mask & 1) : ((T.lo_mask >> 2) & 1);
    if (W[0].nkt_x != xkt || W[0].nkt_h != 4) { set_error("gru_layer_tc: weight / operand k-tile mismatch"); return PB_ERR_STATE; }
    static const bool use_layer = !(getenv("PB_GRU_LAYER") && atoi(getenv("PB_GRU_LAYER")) == 0);
    if (use_layer) {
        static bool la = false;
        if (!la) { PB_CUDA(cudaFuncSetAttribute(tc::k_gru_layer, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::PSMEM_BYTES)); la = true; }
        tc::k_gru_layer<<<(unsigned) (2 * Mt), tc::PG_THREADS, tc::PSMEM_BYTES, st>>>(G);    // one CTA per (direction, row tile), no h exchange
        PB_CUDA(cudaGetLastError());
    } else {
        tc::k_gru_cluster<<<(unsigned) (4 * Mt), tc::THREADS, tc::CSMEM_BYTES, st>>>(G);      // A/B fallback (PB_GRU_LAYER=0): clusters of 2 CTAs
        PB_CUDA(cudaGetLastError());
    }
    N->launches++;
    return PB_OK;
}

int polish_forward_tc(pb_polish_net *N, const uint8_t *d_images, int64_t B, int64_t n_total, int64_t b0, float *d_hidden_dbg,
                      cudaStream_t st) {
    TcPolish &T = *N->tc;
    const int64_t Mt = ceil_div(B, 128);
    const int64_t seq = Mt * PWIN * 8 * TILE_ELEMS;
    PB_TRY(T.img_op.reserve((size_t) (Mt * PWIN * TILE_ELEMS) * 2));
    PB_TRY(T.yenc_hi.reserve((size_t) seq * 2)); PB_TRY(T.yenc_lo.reserve((size_t) seq * 2));
    PB_TRY(T.ydec_hi.reserve((size_t) seq * 2)); PB_TRY(T.ydec_lo.reserve((size_t) seq * 2));
    PB_TRY(T.zero.reserve((size_t) 4 * TILE_ELEMS * 2));
    PB_CUDA(cudaMemsetAsync(T.zero.p, 0, (size_t) 4 * TILE_ELEMS * 2, st));
    for (int w = 0; w < 19; w++) {
        const int i = w * 50;
        k_tc_pack_polish<<<(unsigned) ceil_div(Mt * 128 * PWIN * 4, 256), 256, 0, st>>>(d_images, T.img_op.as<bf16>(), B, i);
        N->launches++;
        // encoder: h0 = carried state (decoder's final state of the previous window, zeros for the first)
        PB_TRY(gru_layer_tc(N, T.enc, N->enc, T.img_op.as<bf16>(), nullptr, 1, w == 0 ? T.zero.as<bf16>() : T.ydec_hi.as<bf16>(),
                            w == 0 ? T.zero.as<bf16>() : T.ydec_lo.as<bf16>(), w != 0, T.yenc_hi.as<bf16>(), T.yenc_lo.as<bf16>(), B, st));
        // decoder: h0 = encoder's final state
        PB_TRY(gru_layer_tc(N, T.dec, N->dec, T.yenc_hi.as<bf16>(), T.yenc_lo.as<bf16>(), 8, T.yenc_hi.as<bf16>(), T.yenc_lo.as<bf16>(), true,
                            T.ydec_hi.as<bf16>(), T.ydec_lo.as<bf16>(), B, st));
        if (d_hidden_dbg) {
            k_tc_unpack_hidden<<<(unsigned) ceil_div(B * 2 * PH, 256), 256, 0, st>>>(T.ydec_hi.as<bf16>(), T.ydec_lo.as<bf16>(),
                                                                                    d_hidden_dbg + ((int64_t) w * n_total + b0) * 2 * PH, B);
            N->launches++;
        }
        k_polish_dense_tiles<<<(unsigned) (Mt * PWIN), 128, 0, st>>>(T.ydec_hi.as<bf16>(), T.ydec_lo.as<bf16>(), N->dW.as<float>(), N->dB.as<float>(),
                                                                    N->acc.as<float>(), B, i);
        N->launches++;
    }
    PB_CUDA(cudaGetLastError());
    return PB_OK;
}

}  // namespace pb

// ------------------------------------------------------------------------------------------------- self test
// C[M][N] = A[M][K] W[N][K]^T + bias through the tcgen05 kernel (EPI_BIAS, fp32 output).  N % 256 == 0, K % 32 == 0.
// variant_images = false: unscaled fp16 images, three products.  true: the variant network's images (tc_upload_lin with_f8),
// a_lo x w_hi where `lo`, corrections in e4m3 where `f8`.
static int test_tc_gemm(int M, int N, int K, const float *h_A, const float *h_W, const float *h_bias, float *h_out, bool variant_images, int lo, int f8) {
    if (N % 256 || K % 32 || M <= 0) { set_error("pb_test_tc_gemm: N %% 256 and K %% 32 must be 0"); return PB_ERR_ARG; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) { set_error("no CUDA device: libpepper_b200 has no CPU fallback"); return PB_ERR_CUDA; }
    const int64_t Mt = ceil_div(M, 128);
    std::vector<uint16_t> ahi, alo;
    F8Tiles a8{{}, {}, 1.f, tc::F8_LO_SCALE};
    tile_matrix(h_A, M, K, Mt * 128, K, ahi, alo, 128, 1.f, &a8);
    TcLin W;
    DevBuf dahi, dalo, da8hi, da8lo, dbias, dout;
    PB_TRY(upload_tiles(dahi, dalo, ahi, alo));
    PB_TRY(upload_f8(da8hi, da8lo, a8));
    PB_TRY(upload_weight(h_W, N, K, N, K, variant_images, W.w_hi, W.w_lo, W.w8_hi, W.w8_lo, W.acc_scale));
    PB_TRY(dbias.reserve(sizeof(float) * N));
    PB_TRY(dout.reserve(sizeof(float) * (size_t) M * N));
    PB_CUDA(cudaMemcpy(dbias.p, h_bias, sizeof(float) * N, cudaMemcpyHostToDevice));
    Args A;
    A.M = M; A.N = N; A.c_ld = 0;
    Dir D = empty_dir();
    Seg &S = D.seg[0];
    S.hi = dahi.as<bf16>();
    if (variant_images && f8) { S.hi8 = da8hi.as<uint8_t>(); S.lo8 = lo ? da8lo.as<uint8_t>() : nullptr; }
    else S.lo = (!variant_images || lo) ? dalo.as<bf16>() : nullptr;
    S.mt_stride = (int64_t) (K / 32) * TILE_ELEMS; S.nkt = K / 32;
    D.w_hi = W.w_hi.as<bf16>(); D.w_lo = W.w_lo.as<bf16>(); D.w8_hi = W.w8_hi.as<uint8_t>(); D.w8_lo = W.w8_lo.as<uint8_t>();
    D.acc_scale = W.acc_scale; D.w_nkt = K / 32;
    D.bias = dbias.as<float>();
    D.y_f32 = dout.as<float>(); D.ldy = N;
    A.d[0] = D; A.d[1] = D;
    PB_TRY(launch_tc<tc::EPI_BIAS>(A, (int) Mt, N / 128, 1, 0));
    PB_CUDA(cudaGetLastError());
    PB_CUDA(cudaDeviceSynchronize());
    PB_CUDA(cudaMemcpy(h_out, dout.p, sizeof(float) * (size_t) M * N, cudaMemcpyDeviceToHost));
    DevBuf *bufs[] = {&dahi, &dalo, &da8hi, &da8lo, &W.w_hi, &W.w_lo, &W.w8_hi, &W.w8_lo, &dbias, &dout};
    for (auto *b : bufs) b->release();
    return PB_OK;
}
extern "C" int pb_test_tc_gemm(int M, int N, int K, const float *h_A, const float *h_W, const float *h_bias, float *h_out) {
    return test_tc_gemm(M, N, K, h_A, h_W, h_bias, h_out, false, 1, 0);
}
extern "C" int pb_test_tc_gemm_f8(int M, int N, int K, const float *h_A, const float *h_W, const float *h_bias, float *h_out, int lo, int f8) {
    return test_tc_gemm(M, N, K, h_A, h_W, h_bias, h_out, true, lo, f8);
}
