// Recurrent-network inference for sm_100a: variant bi-LSTM x2 + MLP head, polish bi-GRU x2 + Linear with
// the 19-window sliding loop.
//
// Design (B200-first, not a translation of the reference's cuDNN/cuBLAS calls through torch):
//  * every recurrent time step is ONE batched GEMM  [B, Kx+Kh] x [Kx+Kh, 4H]  over ALL candidates / images
//    of the chunk, with the input projection (x_t W_ih^T) and the recurrent product (h W_hh^T) fused into the
//    same K loop and the LSTM / GRU cell fused into the epilogue (gates never reach HBM).  Weight rows are
//    re-packed so that the 4 gate pre-activations of one hidden unit are adjacent columns and land in ONE
//    thread's registers; the GRU's n gate keeps its x-part and h-part in separate columns
//    (n = tanh(W_in x + b_in + r * (W_hn h + b_hn)), pepper simple_model.py:12 -> torch.nn.GRU semantics).
//  * both directions of a bidirectional layer run in the same launch (blockIdx.z);
//  * the MLP head is the same GEMM with a bias+SELU epilogue; 512->3 + softmax is a warp-per-row kernel;
//  * polish: Linear(256->5) + softmax + window accumulate is one warp-per-column kernel per window, argmax +
//    phred one kernel at the end (predict_distributed_cpu.py:77-90).
#include "handles.cuh"
#include <stdlib.h>
#include <vector>
#include <algorithm>
#include <math.h>

namespace pb {

constexpr int GBM = 128, GBN = 128, GBK = 16, GTHREADS = 256;
constexpr int GSTRIDE = GBM + 4;     // padded smem row stride (floats)

enum { MODE_BIAS = 0, MODE_SELU = 1, MODE_LSTM = 2, MODE_GRU = 3 };
enum { A_F32 = 0, A_I8 = 1, A_U8 = 2 };

struct GemmDir {
    const void *a0; int64_t lda0;          // first K-segment: [M] rows, K0 valid columns (padded to K0p with zeros)
    const float *a1; int64_t lda1;         // second K-segment (h_prev), K1 columns
    const float *W;                        // [N][Kp] packed, zero padded
    const float *bias;                     // [N]
    float *out; int64_t ldo;               // MODE_BIAS / MODE_SELU: C[M][ldo]
    const float *h_prev; float *h_next; float *c;   // [M][H]
    float *y; int64_t ldy;                 // y[b*ldy + j] = h_new  (pointer already offset by time/direction)
};
struct GemmArgs {
    GemmDir d[2];
    int M, N, K0, K0p, K1, Kp, H, a0_type;
};

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float seluf_(float x) {
    const float alpha = 1.6732632423543772848170429916717f, scale = 1.0507009873554804934193349852946f;
    return x > 0.f ? scale * x : scale * alpha * (expf(x) - 1.0f);
}

// 4 consecutive k of row `row` of the concatenated A operand
template <int A0_TYPE>
__device__ __forceinline__ float4 load_a4(const GemmDir &D, const GemmArgs &G, int row, int k) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row >= G.M) return v;
    if (k < G.K0p) {
        if (A0_TYPE == A_F32 && ((G.K0 & 3) == 0)) {
            if (k < G.K0) v = __ldg(reinterpret_cast<const float4 *>(static_cast<const float *>(D.a0) + (int64_t) row * D.lda0 + k));
        } else {
            float t[4];
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int kk = k + i;
                float x = 0.f;
                if (kk < G.K0) {
                    if (A0_TYPE == A_F32) x = __ldg(static_cast<const float *>(D.a0) + (int64_t) row * D.lda0 + kk);
                    else if (A0_TYPE == A_I8) x = (float) __ldg(static_cast<const int8_t *>(D.a0) + (int64_t) row * D.lda0 + kk);
                    else x = (float) __ldg(static_cast<const uint8_t *>(D.a0) + (int64_t) row * D.lda0 + kk);
                }
                t[i] = x;
            }
            v = make_float4(t[0], t[1], t[2], t[3]);
        }
    } else {
        const int k1 = k - G.K0p;
        if (k1 < G.K1) v = __ldg(reinterpret_cast<const float4 *>(D.a1 + (int64_t) row * D.lda1 + k1));
    }
    return v;
}

template <int MODE, int A0_TYPE>
__global__ void __launch_bounds__(GTHREADS, 2) k_gemm_fused(GemmArgs G) {
    __shared__ __align__(16) float As[2][GBK][GSTRIDE];
    __shared__ __align__(16) float Ws[2][GBK][GSTRIDE];
    const GemmDir &D = G.d[blockIdx.z];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.x * GBM, n0 = blockIdx.y * GBN;
    // loader mapping: 4 lanes cover the 16 k of one row
    const int lr = tid >> 2, lk = (tid & 3) * 4;

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j] = 0.f;

    const int nk = G.Kp / GBK;
    float4 ra[2], rw[2];
    auto gload = [&](int kt) {
        const int k = kt * GBK + lk;
#pragma unroll
        for (int h = 0; h < 2; h++) {
            ra[h] = load_a4<A0_TYPE>(D, G, m0 + lr + 64 * h, k);
            const int n = n0 + lr + 64 * h;
            rw[h] = (n < G.N) ? __ldg(reinterpret_cast<const float4 *>(D.W + (int64_t) n * G.Kp + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto sstore = [&](int buf) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int r = lr + 64 * h;
            As[buf][lk + 0][r] = ra[h].x; As[buf][lk + 1][r] = ra[h].y; As[buf][lk + 2][r] = ra[h].z; As[buf][lk + 3][r] = ra[h].w;
            Ws[buf][lk + 0][r] = rw[h].x; Ws[buf][lk + 1][r] = rw[h].y; Ws[buf][lk + 2][r] = rw[h].z; Ws[buf][lk + 3][r] = rw[h].w;
        }
    };
    gload(0);
    sstore(0);
    __syncthreads();
    for (int kt = 0; kt < nk; kt++) {
        const int buf = kt & 1;
        if (kt + 1 < nk) gload(kt + 1);
#pragma unroll
        for (int k = 0; k < GBK; k++) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[buf][k][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4 *>(&As[buf][k][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Ws[buf][k][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4 *>(&Ws[buf][k][64 + tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
                for (int j = 0; j < 8; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (kt + 1 < nk) {
            sstore(buf ^ 1);
            __syncthreads();
        }
    }

    // ------------------------------------------------------------------ epilogue
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int row = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (row >= G.M) continue;
#pragma unroll
        for (int half = 0; half < 2; half++) {
            const int col = n0 + half * 64 + tx * 4;
            if (col >= G.N) continue;
            const float4 bz = __ldg(reinterpret_cast<const float4 *>(D.bias + col));
            const float v0 = acc[i][half * 4 + 0] + bz.x, v1 = acc[i][half * 4 + 1] + bz.y;
            const float v2 = acc[i][half * 4 + 2] + bz.z, v3 = acc[i][half * 4 + 3] + bz.w;
            if (MODE == MODE_BIAS) {
                *reinterpret_cast<float4 *>(D.out + (int64_t) row * D.ldo + col) = make_float4(v0, v1, v2, v3);
            } else if (MODE == MODE_SELU) {
                *reinterpret_cast<float4 *>(D.out + (int64_t) row * D.ldo + col) = make_float4(seluf_(v0), seluf_(v1), seluf_(v2), seluf_(v3));
            } else if (MODE == MODE_LSTM) {
                // columns: i, f, g, o of hidden unit j  (torch.nn.LSTM gate order, simple_model.py:23)
                const int j = col >> 2;
                const int64_t sidx = (int64_t) row * G.H + j;
                const float ig = sigmoidf_(v0), fg = sigmoidf_(v1), gg = tanhf(v2), og = sigmoidf_(v3);
                const float cn = fg * D.c[sidx] + ig * gg;
                const float hn = og * tanhf(cn);
                D.c[sidx] = cn;
                D.h_next[sidx] = hn;
                D.y[(int64_t) row * D.ldy + j] = hn;
            } else {
                // columns: r, z, n_x, n_h of hidden unit j  (torch.nn.GRU, gate order r,z,n)
                const int j = col >> 2;
                const int64_t sidx = (int64_t) row * G.H + j;
                const float r = sigmoidf_(v0), z = sigmoidf_(v1);
                const float n = tanhf(v2 + r * v3);
                const float hp = D.h_prev[sidx];
                const float hn = (1.0f - z) * n + z * hp;
                D.h_next[sidx] = hn;
                D.y[(int64_t) row * D.ldy + j] = hn;
            }
        }
    }
}

// ------------------------------------------------------------------ small kernels
// variant head: logits = W[3][512] x + b, softmax (simple_model.py:76-82); one warp per candidate.  With a record sink the
// warp also assembles the candidate's 84-byte prediction record (probabilities + the encoder's columns) in place, so the
// buffer a gather sends is produced by the network itself.
__global__ void k_variant_out(const float *__restrict__ x, const float *__restrict__ W, const float *__restrict__ b,
                              float *__restrict__ probs, int64_t n, pb::OutSink S) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t) blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    for (int k = lane; k < 512; k += 32) {
        const float v = x[row * 512 + k];
        s0 = fmaf(v, __ldg(W + k), s0); s1 = fmaf(v, __ldg(W + 512 + k), s1); s2 = fmaf(v, __ldg(W + 1024 + k), s2);
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, d); s1 += __shfl_xor_sync(0xffffffffu, s1, d); s2 += __shfl_xor_sync(0xffffffffu, s2, d);
    }
    s0 += b[0]; s1 += b[1]; s2 += b[2];
    const float m = fmaxf(s0, fmaxf(s1, s2));
    const float e0 = expf(s0 - m), e1 = expf(s1 - m), e2 = expf(s2 - m);
    const float inv = 1.0f / (e0 + e1 + e2);
    if (lane == 0) { probs[row * 3 + 0] = e0 * inv; probs[row * 3 + 1] = e1 * inv; probs[row * 3 + 2] = e2 * inv; }
    if (S.records) {
        pb_pred_record_t *r = S.records + row;
        if (lane == 0) {
            r->probs[0] = e0 * inv; r->probs[1] = e1 * inv; r->probs[2] = e2 * inv;
            r->position = (int32_t) S.cols.positions[row];
            r->region = S.cols.region_of[row];
            r->depth = S.cols.depths[row]; r->freq = S.cols.freqs[row];
        } else {
            // lanes 1..31: two key bytes each (62 = 31 x 2); the key field starts at byte 22 of the 84-byte record
            const uint16_t kb = *reinterpret_cast<const uint16_t *>(S.cols.keys + row * PB_ALLELE_STRIDE + 2 * (lane - 1));
            *reinterpret_cast<uint16_t *>(r->key + 2 * (lane - 1)) = kb;
        }
    }
}

// polish: dense1 (256->5) + softmax, accumulated into acc[b][i+t][5] (predict_distributed_cpu.py:62-81)
__global__ void k_polish_dense_acc(const float *__restrict__ y, const float *__restrict__ W, const float *__restrict__ bias,
                                   float *__restrict__ acc, int64_t n_img, int win_start) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t) blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);   // b*100 + t
    if (row >= n_img * 100) return;
    float s[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int k = lane; k < 256; k += 32) {
        const float v = y[row * 256 + k];
#pragma unroll
        for (int c = 0; c < 5; c++) s[c] = fmaf(v, __ldg(W + c * 256 + k), s[c]);
    }
#pragma unroll
    for (int c = 0; c < 5; c++)
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) s[c] += __shfl_xor_sync(0xffffffffu, s[c], d);
    if (lane == 0) {
        float m = -INFINITY;
#pragma unroll
        for (int c = 0; c < 5; c++) { s[c] += bias[c]; m = fmaxf(m, s[c]); }
        float e[5], sum = 0.f;
#pragma unroll
        for (int c = 0; c < 5; c++) { e[c] = expf(s[c] - m); sum += e[c]; }
        const int64_t b = row / 100;
        const int t = (int) (row - b * 100);
        float *dst = acc + (b * 1000 + win_start + t) * 5;
#pragma unroll
        for (int c = 0; c < 5; c++) dst[c] += e[c] / sum;
    }
}

// torch.max(acc, 2) (first maximal index) and phred = -10 log10(1 - v/count), inf -> 100,
// count = 2 on columns [50, 950) else 1 (predict_distributed_cpu.py:83-90); stored as uint8 (DataStorePredict.py:49)
__global__ void k_polish_finalize(const float *__restrict__ acc, uint8_t *__restrict__ bases, uint8_t *__restrict__ phred, int64_t n_img) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_img * 1000) return;
    const float *a = acc + i * 5;
    int best = 0; float bv = a[0];
#pragma unroll
    for (int c = 1; c < 5; c++) if (a[c] > bv) { bv = a[c]; best = c; }
    const int col = (int) (i % 1000);
    const float count = (col >= 50 && col < 950) ? 2.0f : 1.0f;
    float ph = -10.0f * log10f(1.0f - bv / count);
    if (isinf(ph)) ph = 100.0f;
    bases[i] = (uint8_t) best;
    // numpy astype(uint8) of a float: truncation toward zero (negative / NaN values are implementation defined there)
    phred[i] = (uint8_t) (int) fmaxf(0.f, fminf(ph, 255.f));
}

__global__ void k_copy_hidden(const float *__restrict__ h_dirs /* [2][B][H] */, float *__restrict__ out /* [B][2][H] */, int64_t B, int H) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * B * H) return;
    const int j = (int) (i % H);
    const int64_t b = (i / H) % B;
    const int d = (int) (i / (H * B));
    out[(b * 2 + d) * H + j] = h_dirs[i];
}

// ------------------------------------------------------------------ host helpers
static int round_up(int x, int m) { return (x + m - 1) / m * m; }

struct PackedRnn {      // one direction of one layer
    std::vector<float> W, bias;
    int K0, K0p, K1, Kp, H;
};

// PyTorch LSTM params (gate order i,f,g,o) -> rows 4j+g, K = [x | pad | h | pad]
static PackedRnn pack_lstm(const float *w_ih, const float *w_hh, const float *b_ih, const float *b_hh, int In, int H) {
    PackedRnn P;
    P.K0 = In; P.K0p = round_up(In, 4); P.K1 = H; P.Kp = round_up(P.K0p + H, GBK); P.H = H;
    P.W.assign((size_t) 4 * H * P.Kp, 0.f);
    P.bias.assign((size_t) 4 * H, 0.f);
    for (int j = 0; j < H; j++)
        for (int g = 0; g < 4; g++) {
            float *row = &P.W[(size_t) (4 * j + g) * P.Kp];
            const int src = g * H + j;
            for (int k = 0; k < In; k++) row[k] = w_ih[(size_t) src * In + k];
            for (int k = 0; k < H; k++) row[P.K0p + k] = w_hh[(size_t) src * H + k];
            P.bias[4 * j + g] = b_ih[src] + b_hh[src];
        }
    return P;
}
// PyTorch GRU params (gate order r,z,n) -> rows 4j+{r, z, n_x, n_h}
static PackedRnn pack_gru(const float *w_ih, const float *w_hh, const float *b_ih, const float *b_hh, int In, int H) {
    PackedRnn P;
    P.K0 = In; P.K0p = round_up(In, 4); P.K1 = H; P.Kp = round_up(P.K0p + H, GBK); P.H = H;
    P.W.assign((size_t) 4 * H * P.Kp, 0.f);
    P.bias.assign((size_t) 4 * H, 0.f);
    for (int j = 0; j < H; j++) {
        for (int g = 0; g < 2; g++) {
            float *row = &P.W[(size_t) (4 * j + g) * P.Kp];
            const int src = g * H + j;
            for (int k = 0; k < In; k++) row[k] = w_ih[(size_t) src * In + k];
            for (int k = 0; k < H; k++) row[P.K0p + k] = w_hh[(size_t) src * H + k];
            P.bias[4 * j + g] = b_ih[src] + b_hh[src];
        }
        const int src = 2 * H + j;
        float *rx = &P.W[(size_t) (4 * j + 2) * P.Kp], *rh = &P.W[(size_t) (4 * j + 3) * P.Kp];
        for (int k = 0; k < In; k++) rx[k] = w_ih[(size_t) src * In + k];
        for (int k = 0; k < H; k++) rh[P.K0p + k] = w_hh[(size_t) src * H + k];
        P.bias[4 * j + 2] = b_ih[src];
        P.bias[4 * j + 3] = b_hh[src];
    }
    return P;
}


static int upload_rnn(DevRnn &d, const PackedRnn &p) {
    d.K0 = p.K0; d.K0p = p.K0p; d.K1 = p.K1; d.Kp = p.Kp; d.H = p.H;
    PB_TRY(d.W.reserve(p.W.size() * sizeof(float)));
    PB_TRY(d.bias.reserve(p.bias.size() * sizeof(float)));
    PB_CUDA(cudaMemcpy(d.W.p, p.W.data(), p.W.size() * sizeof(float), cudaMemcpyHostToDevice));
    PB_CUDA(cudaMemcpy(d.bias.p, p.bias.data(), p.bias.size() * sizeof(float), cudaMemcpyHostToDevice));
    return PB_OK;
}
static int upload_lin(DevLin &d, const float *w, const float *b, int N, int K) {
    d.N = N; d.K = K; d.Kp = round_up(K, GBK);
    std::vector<float> W((size_t) N * d.Kp, 0.f);
    for (int n = 0; n < N; n++) memcpy(&W[(size_t) n * d.Kp], w + (size_t) n * K, sizeof(float) * K);
    PB_TRY(d.W.reserve(W.size() * sizeof(float)));
    PB_TRY(d.bias.reserve(sizeof(float) * std::max(N, 4)));
    PB_CUDA(cudaMemcpy(d.W.p, W.data(), W.size() * sizeof(float), cudaMemcpyHostToDevice));
    PB_CUDA(cudaMemcpy(d.bias.p, b, sizeof(float) * N, cudaMemcpyHostToDevice));
    return PB_OK;
}

template <int MODE, int A0_TYPE>
static void launch_gemm(const GemmArgs &G, int ndir, cudaStream_t st) {
    dim3 grid((unsigned) ceil_div(G.M, GBM), (unsigned) ceil_div(G.N, GBN), (unsigned) ndir);
    k_gemm_fused<MODE, A0_TYPE><<<grid, GTHREADS, 0, st>>>(G);
}

}  // namespace pb

using namespace pb;

// =====================================================================================================
// Variant network
// =====================================================================================================
static const char *VARIANT_PARAMS[PB_VARIANT_NET_N_PARAMS] = {
    "encoder.weight_ih_l0", "encoder.weight_hh_l0", "encoder.bias_ih_l0", "encoder.bias_hh_l0",
    "encoder.weight_ih_l0_reverse", "encoder.weight_hh_l0_reverse", "encoder.bias_ih_l0_reverse", "encoder.bias_hh_l0_reverse",
    "decoder.weight_ih_l0", "decoder.weight_hh_l0", "decoder.bias_ih_l0", "decoder.bias_hh_l0",
    "decoder.weight_ih_l0_reverse", "decoder.weight_hh_l0_reverse", "decoder.bias_ih_l0_reverse", "decoder.bias_hh_l0_reverse",
    "linear_1.weight", "linear_1.bias", "linear_2.weight", "linear_2.bias", "linear_3.weight", "linear_3.bias",
    "linear_4.weight", "linear_4.bias", "linear_5.weight", "linear_5.bias", "output_layer_type.weight", "output_layer_type.bias"};
static const int64_t VARIANT_NUMEL[PB_VARIANT_NET_N_PARAMS] = {
    1024 * 26, 1024 * 256, 1024, 1024, 1024 * 26, 1024 * 256, 1024, 1024,
    1024 * 512, 1024 * 256, 1024, 1024, 1024 * 512, 1024 * 256, 1024, 1024,
    512 * 16896, 512, 512 * 512, 512, 512 * 512, 512, 512 * 512, 512, 512 * 512, 512, 3 * 512, 3};

extern "C" const char *pb_variant_net_param_name(int i) { return (i >= 0 && i < PB_VARIANT_NET_N_PARAMS) ? VARIANT_PARAMS[i] : nullptr; }
extern "C" int64_t pb_variant_net_param_numel(int i) { return (i >= 0 && i < PB_VARIANT_NET_N_PARAMS) ? VARIANT_NUMEL[i] : -1; }


constexpr int VT = 33, VH = 256;
constexpr int64_t VARIANT_CHUNK = 9472;     // 74 row tiles: 74 x 8 x 2 CTAs = 4 full waves of 2 CTAs x 148 SMs per LSTM step

extern "C" int pb_variant_net_create(pb_variant_net_t **out, int device, const float *const *P) {
    if (!out || !P) { set_error("null argument"); return PB_ERR_ARG; }
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= device) {
        set_error("no CUDA device %d (found %d): libpepper_b200 has no CPU fallback", device, n);
        return PB_ERR_CUDA;
    }
    for (int i = 0; i < PB_VARIANT_NET_N_PARAMS; i++) if (!P[i]) { set_error("missing parameter %s", VARIANT_PARAMS[i]); return PB_ERR_ARG; }
    PB_CUDA(cudaSetDevice(device));
    auto *N = new pb_variant_net();
    N->device = device;
    N->tc = new TcVariant();
    for (int d = 0; d < 2; d++) {
        const PackedRnn pe = pack_lstm(P[4 * d + 0], P[4 * d + 1], P[4 * d + 2], P[4 * d + 3], 26, VH);
        const PackedRnn pd = pack_lstm(P[8 + 4 * d + 0], P[8 + 4 * d + 1], P[8 + 4 * d + 2], P[8 + 4 * d + 3], 512, VH);
        PB_TRY(upload_rnn(N->enc[d], pe));
        PB_TRY(upload_rnn(N->dec[d], pd));
        PB_TRY(tc_upload_rnn(N->tc->enc[d], pe.W.data(), pe.K0, pe.K0p, VH, pe.Kp, true));
        PB_TRY(tc_upload_rnn(N->tc->dec[d], pd.W.data(), pd.K0, pd.K0p, VH, pd.Kp, true));
    }
    PB_TRY(upload_lin(N->lin[0], P[16], P[17], 512, VT * 512));
    PB_TRY(tc_upload_lin(N->tc->lin[0], P[16], 512, VT * 512, true));
    for (int i = 1; i < 5; i++) {
        PB_TRY(upload_lin(N->lin[i], P[16 + 2 * i], P[17 + 2 * i], 512, 512));
        PB_TRY(tc_upload_lin(N->tc->lin[i], P[16 + 2 * i], 512, 512, true));
    }
    PB_TRY(upload_lin(N->outl, P[26], P[27], 3, 512));
    *out = N;
    return PB_OK;
}

extern "C" int pb_variant_net_destroy(pb_variant_net_t *N) {
    if (!N) return PB_OK;
    for (int d = 0; d < 2; d++) { N->enc[d].W.release(); N->enc[d].bias.release(); N->dec[d].W.release(); N->dec[d].bias.release(); }
    for (auto &l : N->lin) { l.W.release(); l.bias.release(); }
    N->outl.W.release(); N->outl.bias.release();
    DevBuf *bufs[] = {&N->h[0], &N->h[1], &N->c, &N->yenc, &N->ydec, &N->l[0], &N->l[1], &N->img, &N->probs};
    for (auto *b : bufs) b->release();
    if (N->tc) {
        TcVariant &T = *N->tc;
        for (int d = 0; d < 2; d++)
            for (TcRnn *r : {&T.enc[d], &T.dec[d]}) { r->w_hi.release(); r->w_lo.release(); r->w8_hi.release(); r->w8_lo.release(); }
        for (auto &l : T.lin) { l.w_hi.release(); l.w_lo.release(); l.w8_hi.release(); l.w8_lo.release(); }
        DevBuf *tb[] = {&T.img_op, &T.yenc_hi, &T.yenc_lo, &T.ydec_hi, &T.ydec_lo, &T.c, &T.act_hi[0], &T.act_hi[1], &T.act_lo[0], &T.act_lo[1], &T.final_f32,
                        &T.img_op8, &T.yenc_hi8, &T.yenc_lo8, &T.ydec_hi8, &T.ydec_lo8, &T.act_hi8[0], &T.act_hi8[1], &T.act_lo8[0], &T.act_lo8[1]};
        for (auto *b : tb) b->release();
        delete N->tc;
    }
    delete N;
    return PB_OK;
}

extern "C" int pb_variant_net_set_mode(pb_variant_net_t *N, int mode) {
    if (!N) return PB_ERR_ARG;
    if (mode != 0 && mode != 1) { set_error("mode %d unknown (0 = fp32 FFMA, 1 = tcgen05 bf16x3)", mode); return PB_ERR_ARG; }
    N->mode = mode;
    return PB_OK;
}
// experiments (DESIGN.md "two-product variant"): which GEMMs keep the third tensor-core product
extern "C" int pb_variant_net_set_lo_mask(pb_variant_net_t *N, int mask) {
    if (!N || !N->tc) { set_error("no tcgen05 state"); return PB_ERR_ARG; }
    N->tc->lo_mask = mask & 0x1f;
    return PB_OK;
}
// which GEMMs run their correction products as e4m3 MMAs (same bits; 0 = the fp16 split everywhere)
extern "C" int pb_variant_net_set_f8_mask(pb_variant_net_t *N, int mask) {
    if (!N || !N->tc) { set_error("no tcgen05 state"); return PB_ERR_ARG; }
    N->tc->f8_mask = mask & 0x1f;
    return PB_OK;
}
extern "C" int pb_polish_net_set_lo_mask(pb_polish_net_t *N, int mask) {
    if (!N || !N->tc) { set_error("no tcgen05 state"); return PB_ERR_ARG; }
    N->tc->lo_mask = mask & 0x7;
    return PB_OK;
}
extern "C" int pb_variant_net_launches(pb_variant_net_t *N, int64_t *n) {
    if (!N || !n) return PB_ERR_ARG;
    *n = N->launches;
    return PB_OK;
}

static void launch_variant_out(const float *x, const float *W, const float *b, float *probs, int64_t n, const pb::OutSink &S, cudaStream_t st) {
    k_variant_out<<<(unsigned) ceil_div(n, 8), 256, 0, st>>>(x, W, b, probs, n, S);
}

static int variant_reserve(pb_variant_net *N, int64_t B) {
    if (B <= N->chunk) return PB_OK;
    for (int i = 0; i < 2; i++) PB_TRY(N->h[i].reserve(sizeof(float) * 2 * B * VH));
    PB_TRY(N->c.reserve(sizeof(float) * 2 * B * VH));
    PB_TRY(N->yenc.reserve(sizeof(float) * B * VT * 512));
    PB_TRY(N->ydec.reserve(sizeof(float) * B * VT * 512));
    for (int i = 0; i < 2; i++) PB_TRY(N->l[i].reserve(sizeof(float) * B * 512));
    N->chunk = B;
    return PB_OK;
}

// one bidirectional LSTM layer over T steps. x: a0 source (int8 images or fp32 sequence), row stride lda0 per candidate,
// feature stride `xstep` per time step
template <int A0_TYPE>
static int lstm_layer(pb_variant_net *N, DevRnn *L, const void *x, int64_t lda0, int64_t xstep_bytes, int K0, int64_t B,
                      float *y /* [B][T][512] */, cudaStream_t st) {
    PB_CUDA(cudaMemsetAsync(N->h[0].p, 0, sizeof(float) * 2 * B * VH, st));
    PB_CUDA(cudaMemsetAsync(N->c.p, 0, sizeof(float) * 2 * B * VH, st));
    for (int t = 0; t < VT; t++) {
        GemmArgs G;
        G.M = (int) B; G.N = 4 * VH; G.K0 = K0; G.K0p = L[0].K0p; G.K1 = VH; G.Kp = L[0].Kp; G.H = VH; G.a0_type = A0_TYPE;
        for (int d = 0; d < 2; d++) {
            const int tt = d == 0 ? t : VT - 1 - t;
            GemmDir &D = G.d[d];
            D.a0 = static_cast<const char *>(x) + (int64_t) tt * xstep_bytes; D.lda0 = lda0;
            D.a1 = N->h[t & 1].as<float>() + (int64_t) d * B * VH; D.lda1 = VH;
            D.W = L[d].W.as<float>(); D.bias = L[d].bias.as<float>();
            D.out = nullptr; D.ldo = 0;
            D.h_prev = D.a1; D.h_next = N->h[(t + 1) & 1].as<float>() + (int64_t) d * B * VH;
            D.c = N->c.as<float>() + (int64_t) d * B * VH;
            D.y = y + (int64_t) tt * 512 + d * VH; D.ldy = (int64_t) VT * 512;
        }
        launch_gemm<MODE_LSTM, A0_TYPE>(G, 2, st);
        N->launches++;
    }
    PB_CUDA(cudaGetLastError());
    return PB_OK;
}

static int variant_forward(pb_variant_net_t *N, const int8_t *d_images, int64_t n, float *d_probs, float *d_hidden_dbg,
                           const pb::OutSink &sink, void *stream_);

extern "C" int pb_variant_net_forward_device(pb_variant_net_t *N, const int8_t *d_images, int64_t n, float *d_probs,
                                             float *d_hidden_dbg, void *stream_) {
    return variant_forward(N, d_images, n, d_probs, d_hidden_dbg, pb::OutSink{}, stream_);
}

extern "C" int pb_variant_net_forward_records_device(pb_variant_net_t *N, const int8_t *d_images, int64_t n, float *d_probs,
                                                     const pb_candidate_columns_t *cols, pb_pred_record_t *d_records, void *stream_) {
    pb::OutSink S{};
    if (d_records) {
        if (!cols || !cols->positions || !cols->region_of || !cols->depths || !cols->freqs || !cols->keys) {
            set_error("record sink needs all candidate columns"); return PB_ERR_ARG;
        }
        S.cols = *cols; S.records = d_records;
    }
    return variant_forward(N, d_images, n, d_probs, nullptr, S, stream_);
}

static int variant_forward(pb_variant_net_t *N, const int8_t *d_images, int64_t n, float *d_probs, float *d_hidden_dbg,
                           const pb::OutSink &sink, void *stream_) {
    if (!N || (n > 0 && (!d_images || !d_probs))) { set_error("null argument"); return PB_ERR_ARG; }
    cudaStream_t st = (cudaStream_t) stream_;
    PB_CUDA(cudaSetDevice(N->device));
    N->launches = 0;
    for (int64_t b0 = 0; b0 < n; b0 += VARIANT_CHUNK) {
        const int64_t B = std::min(VARIANT_CHUNK, n - b0);
        const int8_t *img = d_images + b0 * VT * 26;
        if (N->mode >= 1) {
            PB_TRY(variant_forward_tc(N, img, B, d_probs + b0 * 3, d_hidden_dbg ? d_hidden_dbg + b0 * VT * 512 : nullptr, st, launch_variant_out,
                                      sink.at(b0)));
            continue;
        }
        PB_TRY(variant_reserve(N, B));
        PB_TRY(lstm_layer<A_I8>(N, N->enc, img, (int64_t) VT * 26, 26, 26, B, N->yenc.as<float>(), st));
        PB_TRY(lstm_layer<A_F32>(N, N->dec, N->yenc.p, (int64_t) VT * 512, 512 * sizeof(float), 512, B, N->ydec.as<float>(), st));
        if (d_hidden_dbg)
            PB_CUDA(cudaMemcpyAsync(d_hidden_dbg + b0 * VT * 512, N->ydec.p, sizeof(float) * B * VT * 512, cudaMemcpyDeviceToDevice, st));
        // MLP head (simple_model.py:56-75): 5 x (Linear + SELU); dropout is identity in eval
        const float *cur = N->ydec.as<float>();
        int64_t ld = (int64_t) VT * 512;
        for (int i = 0; i < 5; i++) {
            GemmArgs G;
            G.M = (int) B; G.N = 512; G.K0 = N->lin[i].K; G.K0p = N->lin[i].K; G.K1 = 0; G.Kp = N->lin[i].Kp; G.H = 0; G.a0_type = A_F32;
            GemmDir &D = G.d[0];
            D.a0 = cur; D.lda0 = ld; D.a1 = nullptr; D.lda1 = 0; D.W = N->lin[i].W.as<float>(); D.bias = N->lin[i].bias.as<float>();
            D.out = N->l[i & 1].as<float>(); D.ldo = 512;
            D.h_prev = nullptr; D.h_next = nullptr; D.c = nullptr; D.y = nullptr; D.ldy = 0;
            G.d[1] = G.d[0];
            launch_gemm<MODE_SELU, A_F32>(G, 1, st);
            N->launches++;
            cur = N->l[i & 1].as<float>(); ld = 512;
        }
        k_variant_out<<<(unsigned) ceil_div(B, 8), 256, 0, st>>>(cur, N->outl.W.as<float>(), N->outl.bias.as<float>(), d_probs + b0 * 3, B, sink.at(b0));
        N->launches++;
        PB_CUDA(cudaGetLastError());
    }
    return PB_OK;
}

extern "C" int pb_variant_net_forward_host(pb_variant_net_t *N, const int8_t *h_images, int64_t n, float *h_probs,
                                           float *h_hidden_dbg, void *stream_) {
    if (!N) return PB_ERR_ARG;
    cudaStream_t st = (cudaStream_t) stream_;
    PB_CUDA(cudaSetDevice(N->device));
    if (n <= 0) return PB_OK;
    DevBuf hid;
    PB_TRY(N->img.reserve((size_t) n * VT * 26));
    PB_TRY(N->probs.reserve(sizeof(float) * n * 3));
    if (h_hidden_dbg) PB_TRY(hid.reserve(sizeof(float) * n * VT * 512));
    PB_CUDA(cudaMemcpyAsync(N->img.p, h_images, (size_t) n * VT * 26, cudaMemcpyHostToDevice, st));
    int rc = pb_variant_net_forward_device(N, N->img.as<int8_t>(), n, N->probs.as<float>(), h_hidden_dbg ? hid.as<float>() : nullptr, stream_);
    if (rc == PB_OK) {
        cudaError_t e = cudaMemcpyAsync(h_probs, N->probs.p, sizeof(float) * n * 3, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && h_hidden_dbg) e = cudaMemcpyAsync(h_hidden_dbg, hid.p, sizeof(float) * n * VT * 512, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { set_error("variant net copy back: %s", cudaGetErrorString(e)); rc = PB_ERR_CUDA; }
    }
    hid.release();
    return rc;
}

// =====================================================================================================
// Polish network
// =====================================================================================================
static const char *POLISH_PARAMS[PB_POLISH_NET_N_PARAMS] = {
    "gru_encoder.weight_ih_l0", "gru_encoder.weight_hh_l0", "gru_encoder.bias_ih_l0", "gru_encoder.bias_hh_l0",
    "gru_encoder.weight_ih_l0_reverse", "gru_encoder.weight_hh_l0_reverse", "gru_encoder.bias_ih_l0_reverse", "gru_encoder.bias_hh_l0_reverse",
    "gru_decoder.weight_ih_l0", "gru_decoder.weight_hh_l0", "gru_decoder.bias_ih_l0", "gru_decoder.bias_hh_l0",
    "gru_decoder.weight_ih_l0_reverse", "gru_decoder.weight_hh_l0_reverse", "gru_decoder.bias_ih_l0_reverse", "gru_decoder.bias_hh_l0_reverse",
    "dense1.weight", "dense1.bias"};
static const int64_t POLISH_NUMEL[PB_POLISH_NET_N_PARAMS] = {
    384 * 10, 384 * 128, 384, 384, 384 * 10, 384 * 128, 384, 384,
    384 * 256, 384 * 128, 384, 384, 384 * 256, 384 * 128, 384, 384, 5 * 256, 5};
extern "C" const char *pb_polish_net_param_name(int i) { return (i >= 0 && i < PB_POLISH_NET_N_PARAMS) ? POLISH_PARAMS[i] : nullptr; }
extern "C" int64_t pb_polish_net_param_numel(int i) { return (i >= 0 && i < PB_POLISH_NET_N_PARAMS) ? POLISH_NUMEL[i] : -1; }

constexpr int PH = 128, PWIN = 100, PJUMP = 50, PSEQ = 1000, PNWIN = 19;
constexpr int64_t POLISH_CHUNK = 8192;


extern "C" int pb_polish_net_create(pb_polish_net_t **out, int device, const float *const *P) {
    if (!out || !P) { set_error("null argument"); return PB_ERR_ARG; }
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= device) {
        set_error("no CUDA device %d (found %d): libpepper_b200 has no CPU fallback", device, n);
        return PB_ERR_CUDA;
    }
    for (int i = 0; i < PB_POLISH_NET_N_PARAMS; i++) if (!P[i]) { set_error("missing parameter %s", POLISH_PARAMS[i]); return PB_ERR_ARG; }
    PB_CUDA(cudaSetDevice(device));
    auto *N = new pb_polish_net();
    N->device = device;
    N->tc = new TcPolish();
    for (int d = 0; d < 2; d++) {
        const PackedRnn pe = pack_gru(P[4 * d + 0], P[4 * d + 1], P[4 * d + 2], P[4 * d + 3], 10, PH);
        const PackedRnn pd = pack_gru(P[8 + 4 * d + 0], P[8 + 4 * d + 1], P[8 + 4 * d + 2], P[8 + 4 * d + 3], 256, PH);
        PB_TRY(upload_rnn(N->enc[d], pe));
        PB_TRY(upload_rnn(N->dec[d], pd));
        PB_TRY(tc_upload_rnn(N->tc->enc[d], pe.W.data(), pe.K0, pe.K0p, PH, pe.Kp, false));
        PB_TRY(tc_upload_rnn(N->tc->dec[d], pd.W.data(), pd.K0, pd.K0p, PH, pd.Kp, false));
    }
    PB_TRY(N->dW.reserve(sizeof(float) * 5 * 256));
    PB_TRY(N->dB.reserve(sizeof(float) * 8));
    PB_CUDA(cudaMemcpy(N->dW.p, P[16], sizeof(float) * 5 * 256, cudaMemcpyHostToDevice));
    PB_CUDA(cudaMemcpy(N->dB.p, P[17], sizeof(float) * 5, cudaMemcpyHostToDevice));
    *out = N;
    return PB_OK;
}

extern "C" int pb_polish_net_destroy(pb_polish_net_t *N) {
    if (!N) return PB_OK;
    for (int d = 0; d < 2; d++) { N->enc[d].W.release(); N->enc[d].bias.release(); N->dec[d].W.release(); N->dec[d].bias.release(); }
    DevBuf *bufs[] = {&N->dW, &N->dB, &N->h[0], &N->h[1], &N->yenc, &N->ydec, &N->acc, &N->img, &N->bases, &N->phred};
    for (auto *b : bufs) b->release();
    if (N->tc) {
        TcPolish &T = *N->tc;
        for (int d = 0; d < 2; d++) { T.enc[d].w_hi.release(); T.enc[d].w_lo.release(); T.dec[d].w_hi.release(); T.dec[d].w_lo.release(); }
        DevBuf *tb[] = {&T.img_op, &T.yenc_hi, &T.yenc_lo, &T.ydec_hi, &T.ydec_lo, &T.zero, &T.flags};
        for (auto *b : tb) b->release();
        delete N->tc;
    }
    delete N;
    return PB_OK;
}
extern "C" int pb_polish_net_set_mode(pb_polish_net_t *N, int mode) {
    if (!N) return PB_ERR_ARG;
    if (mode != 0 && mode != 1) { set_error("mode %d unknown (0 = fp32 FFMA, 1 = tcgen05 bf16x3)", mode); return PB_ERR_ARG; }
    N->mode = mode;
    return PB_OK;
}
extern "C" int pb_polish_net_launches(pb_polish_net_t *N, int64_t *n) {
    if (!N || !n) return PB_ERR_ARG;
    *n = N->launches;
    return PB_OK;
}

// one bidirectional GRU layer over the 100 steps of a window; h buffers ping-pong, the final state ends in N->h[0]
template <int A0_TYPE>
static int gru_layer(pb_polish_net *N, DevRnn *L, const void *x, int64_t lda0, int64_t xstep_bytes, int K0, int64_t B,
                     float *y /* [B][100][256] */, cudaStream_t st) {
    for (int t = 0; t < PWIN; t++) {
        GemmArgs G;
        G.M = (int) B; G.N = 4 * PH; G.K0 = K0; G.K0p = L[0].K0p; G.K1 = PH; G.Kp = L[0].Kp; G.H = PH; G.a0_type = A0_TYPE;
        for (int d = 0; d < 2; d++) {
            const int tt = d == 0 ? t : PWIN - 1 - t;
            GemmDir &D = G.d[d];
            D.a0 = static_cast<const char *>(x) + (int64_t) tt * xstep_bytes; D.lda0 = lda0;
            D.a1 = N->h[t & 1].as<float>() + (int64_t) d * B * PH; D.lda1 = PH;
            D.W = L[d].W.as<float>(); D.bias = L[d].bias.as<float>();
            D.out = nullptr; D.ldo = 0;
            D.h_prev = D.a1; D.h_next = N->h[(t + 1) & 1].as<float>() + (int64_t) d * B * PH; D.c = nullptr;
            D.y = y + (int64_t) tt * 256 + d * PH; D.ldy = (int64_t) PWIN * 256;
        }
        launch_gemm<MODE_GRU, A0_TYPE>(G, 2, st);
        N->launches++;
    }
    // PWIN is even: the state after the last step is back in h[0]
    PB_CUDA(cudaGetLastError());
    return PB_OK;
}

extern "C" int pb_polish_net_forward_device(pb_polish_net_t *N, const uint8_t *d_images, int64_t n, uint8_t *d_bases,
                                            uint8_t *d_phred, float *d_hidden_dbg, float *d_acc_dbg, void *stream_) {
    if (!N || (n > 0 && (!d_images || !d_bases || !d_phred))) { set_error("null argument"); return PB_ERR_ARG; }
    cudaStream_t st = (cudaStream_t) stream_;
    PB_CUDA(cudaSetDevice(N->device));
    N->launches = 0;
    // tcgen05 mode: a window layer is one cooperative launch of 4 CTAs per 128-image row tile, all resident
    int64_t chunk = POLISH_CHUNK;
    if (N->mode == 1) {
        int sms = 0;
        PB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, N->device));
        // k_gru_layer: one CTA per (direction, row tile) -> sms / 2 row tiles fill the GPU; the pair kernels need 4 CTAs per row tile
        const bool layer = !(getenv("PB_GRU_LAYER") && atoi(getenv("PB_GRU_LAYER")) == 0);
        chunk = std::max<int64_t>(1, sms / (layer ? 2 : 4)) * 128;
    }
    for (int64_t b0 = 0; b0 < n; b0 += chunk) {
        const int64_t B = std::min(chunk, n - b0);
        if (B > N->chunk) {
            if (N->mode == 0) {
                for (int i = 0; i < 2; i++) PB_TRY(N->h[i].reserve(sizeof(float) * 2 * B * PH));
                PB_TRY(N->yenc.reserve(sizeof(float) * B * PWIN * 256));
                PB_TRY(N->ydec.reserve(sizeof(float) * B * PWIN * 256));
            }
            PB_TRY(N->acc.reserve(sizeof(float) * B * PSEQ * 5));
            N->chunk = B;
        }
        const uint8_t *img = d_images + b0 * PSEQ * 10;
        if (N->mode == 0) PB_CUDA(cudaMemsetAsync(N->h[0].p, 0, sizeof(float) * 2 * B * PH, st));       // hidden = zeros (cpu.py:53)
        PB_CUDA(cudaMemsetAsync(N->acc.p, 0, sizeof(float) * B * PSEQ * 5, st));
        if (N->mode == 1) {
            PB_TRY(polish_forward_tc(N, img, B, n, b0, d_hidden_dbg, st));
        } else
        for (int w = 0; w < PNWIN; w++) {
            const int i = w * PJUMP;
            // encoder: h0 = carried hidden; decoder: h0 = encoder's final state; its final state is carried on
            PB_TRY(gru_layer<A_U8>(N, N->enc, img + (int64_t) i * 10, (int64_t) PSEQ * 10, 10, 10, B, N->yenc.as<float>(), st));
            PB_TRY(gru_layer<A_F32>(N, N->dec, N->yenc.p, (int64_t) PWIN * 256, 256 * sizeof(float), 256, B, N->ydec.as<float>(), st));
            if (d_hidden_dbg) {
                k_copy_hidden<<<(unsigned) ceil_div(2 * B * PH, 256), 256, 0, st>>>(N->h[0].as<float>(),
                                                                                 d_hidden_dbg + ((int64_t) w * n + b0) * 2 * PH, B, PH);
                N->launches++;
            }
            k_polish_dense_acc<<<(unsigned) ceil_div(B * PWIN, 8), 256, 0, st>>>(N->ydec.as<float>(), N->dW.as<float>(), N->dB.as<float>(),
                                                                                 N->acc.as<float>(), B, i);
            N->launches++;
        }
        k_polish_finalize<<<(unsigned) ceil_div(B * PSEQ, 256), 256, 0, st>>>(N->acc.as<float>(), d_bases + b0 * PSEQ, d_phred + b0 * PSEQ, B);
        N->launches++;
        if (d_acc_dbg)
            PB_CUDA(cudaMemcpyAsync(d_acc_dbg + b0 * PSEQ * 5, N->acc.p, sizeof(float) * B * PSEQ * 5, cudaMemcpyDeviceToDevice, st));
        PB_CUDA(cudaGetLastError());
    }
    return PB_OK;
}

extern "C" int pb_polish_net_forward_host(pb_polish_net_t *N, const uint8_t *h_images, int64_t n, uint8_t *h_bases,
                                          uint8_t *h_phred, float *h_hidden_dbg, float *h_acc_dbg, void *stream_) {
    if (!N) return PB_ERR_ARG;
    cudaStream_t st = (cudaStream_t) stream_;
    PB_CUDA(cudaSetDevice(N->device));
    if (n <= 0) return PB_OK;
    DevBuf hid, accd;
    PB_TRY(N->img.reserve((size_t) n * PSEQ * 10));
    PB_TRY(N->bases.reserve((size_t) n * PSEQ));
    PB_TRY(N->phred.reserve((size_t) n * PSEQ));
    if (h_hidden_dbg) PB_TRY(hid.reserve(sizeof(float) * PNWIN * n * 2 * PH));
    if (h_acc_dbg) PB_TRY(accd.reserve(sizeof(float) * n * PSEQ * 5));
    PB_CUDA(cudaMemcpyAsync(N->img.p, h_images, (size_t) n * PSEQ * 10, cudaMemcpyHostToDevice, st));
    int rc = pb_polish_net_forward_device(N, N->img.as<uint8_t>(), n, N->bases.as<uint8_t>(), N->phred.as<uint8_t>(),
                                          h_hidden_dbg ? hid.as<float>() : nullptr, h_acc_dbg ? accd.as<float>() : nullptr, stream_);
    if (rc == PB_OK) {
        cudaError_t e = cudaMemcpyAsync(h_bases, N->bases.p, (size_t) n * PSEQ, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_phred, N->phred.p, (size_t) n * PSEQ, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && h_hidden_dbg) e = cudaMemcpyAsync(h_hidden_dbg, hid.p, sizeof(float) * PNWIN * n * 2 * PH, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && h_acc_dbg) e = cudaMemcpyAsync(h_acc_dbg, accd.p, sizeof(float) * n * PSEQ * 5, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { set_error("polish net copy back: %s", cudaGetErrorString(e)); rc = PB_ERR_CUDA; }
    }
    hid.release(); accd.release();
    return rc;
}
