// tcgen05 GEMM with fused LSTM / GRU / SELU epilogues for sm_100a.
//
//   D[128 x 128] (fp32, TMEM)  +=  A[128 x 32] (bf16, smem)  x  B[128 x 32]^T (bf16, smem)      per k-tile
//
// fp32-equivalent precision comes from a bf16 hi/lo split of BOTH operands and three tensor-core products per
// k-tile accumulated into the same TMEM tile:  a*w ~= a_hi*w_hi + a_hi*w_lo + a_lo*w_hi   (error ~2^-16 relative).
//
// Every operand lives in HBM already in the shared-memory image of its tile ("tiled operand": for a tile of 128
// rows x 32 k, element (r, k) sits at  (k/8)*1024 + r*8 + k%8  — the UMMA K-major no-swizzle canonical layout with
// core matrices of 8 rows x 16 B, SBO = 128 B between 8-row groups, LBO = 2048 B between the two 8-element K chunks
// of one MMA).  The producer warp therefore moves whole tiles with cp.async.bulk (TMA engine, no tensor map) onto an
// mbarrier; one elected thread issues tcgen05.mma; tcgen05.commit releases the stage / signals the epilogue; four
// epilogue warps read the accumulator with tcgen05.ld (one TMEM lane = one batch row per thread), apply bias + cell,
// and write the NEXT operand (h_t as bf16 hi/lo tiles) straight from registers, so activations never exist in fp32
// in HBM between layers.
//
// The variant network's persistent kernels (k_tc_gemm_p, k_lstm_layer) can also run the two correction products of a k-tile
// in e4m3 (tcgen05.mma kind::f8f6f4, one K32 MMA = half the tensor time of the two K16 fp16 MMAs it replaces): the main
// product a_hi * w_hi stays fp16 and the corrections, ~2^-12 of it, only need a few significant bits.  See "e4m3 correction
// operands" below.
#pragma once
#include "common.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>

namespace pb {
namespace tc {

// 16-bit operand type of the hi / lo split.  Round 2: fp16 (11 + 11 significant bits: a*w ~= a_hi*w_hi + a_hi*w_lo + a_lo*w_hi is
// good to ~2^-22 relative, 10-50 x closer to the fp32 reference than the bf16 split at the same three products per k-tile —
// scripts/sim_precision.py, DESIGN.md).  Activations are clamped to +-65504 (recurrent states are in [-1, 1]; MLP
// activations of O(1..10)); -DPB_OPERAND_BF16 restores the round-1 bf16 split (8 + 8 bits, no range limit).
#ifdef PB_OPERAND_BF16
typedef __nv_bfloat16 op_t;
constexpr uint32_t OP_FMT = 1u;                      // tcgen05 kind::f16 a_format / b_format: 1 = BF16
__host__ __device__ __forceinline__ uint16_t op_bits(float v) { return __bfloat16_as_ushort(__float2bfloat16_rn(v)); }
__host__ __device__ __forceinline__ float op_val(uint32_t b) { return __bfloat162float(__ushort_as_bfloat16((unsigned short) (b & 0xffffu))); }
#else
typedef __half op_t;
constexpr uint32_t OP_FMT = 0u;                      // 0 = F16
__host__ __device__ __forceinline__ uint16_t op_bits(float v) { return __half_as_ushort(__float2half_rn(fminf(fmaxf(v, -65504.f), 65504.f))); }
__host__ __device__ __forceinline__ float op_val(uint32_t b) { return __half2float(__ushort_as_half((unsigned short) (b & 0xffffu))); }
#endif

constexpr int BM = 128, BN = 128, BK = 32, STAGES = 3;
constexpr int TILE_ELEMS = 128 * BK;                 // 4096 bf16
constexpr int TILE_BYTES = TILE_ELEMS * 2;           // 8192
constexpr int STAGE_BYTES = 4 * TILE_BYTES;          // A_hi, A_lo, B_hi, B_lo
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 128;
constexpr int THREADS = 320;                         // warp 0 producer, warp 1 MMA issuer, warps 2-9 epilogue
constexpr int EPI_COLS = BN / 2;                     // columns per epilogue warp (two warps share a TMEM lane quarter)
constexpr int TMEM_COLS = 128;

enum { EPI_BIAS = 0, EPI_SELU = 1, EPI_LSTM = 2, EPI_GRU = 3 };

struct Seg {                       // one K-segment of the A operand
    const op_t *hi, *lo;  // lo == nullptr: exactly representable operand (int8 images), a_lo*w_hi product skipped
    const uint8_t *hi8, *lo8;      // k_tc_gemm_p: hi8 != nullptr runs the corrections in e4m3 (lo8 == nullptr: without a_lo*w_hi)
    int64_t mt_stride;             // elements between consecutive row tiles
    int nkt;                       // k-tiles in this segment
};
struct Dir {
    Seg seg[2];
    const op_t *w_hi, *w_lo;   // [n_tile][w_nkt][TILE_ELEMS]
    const uint8_t *w8_hi, *w8_lo;       // e4m3 weight images, same tiling (k_tc_gemm_p)
    float acc_scale;                    // accumulator -> GEMM value (2^(E-12) for scaled weight images, else 1)
    int w_nkt;                          // k-tiles per n-tile of the packed weight (>= k-tiles of this launch)
    const float *bias;                  // [N]
    float *c;                           // LSTM cell state [H][c_ld]
    const op_t *hp_hi, *hp_lo; // GRU: previous hidden state as a tiled operand (k-tile = unit/32)
    int64_t hp_mt_stride;
    op_t *y_hi, *y_lo;         // output operand tiles: tile (mt, y_kt0 + col/32); y_lo may be nullptr (k_tc_gemm_p)
    uint8_t *y_hi8, *y_lo8;    // optional e4m3 output images (k_tc_gemm_p)
    int64_t y_mt_stride;
    int y_kt0;
    float *y_f32; int64_t ldy;          // optional fp32 copy  y_f32[row*ldy + col]
};
struct Args {
    Dir d[2];
    int M, N;                           // valid rows; N = columns of the packed weight (multiple of 128)
    int64_t c_ld;
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u) : "memory");
}
// K-major, no swizzle: LBO = 2048 B (K chunk stride), SBO = 128 B (8-row group stride), version 1 (sm_100)
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {
    uint64_t d = 0;
    d |= (uint64_t) ((addr >> 4) & 0x3FFF);
    d |= (uint64_t) ((2048u >> 4) & 0x3FFF) << 16;
    d |= (uint64_t) ((128u >> 4) & 0x3FFF) << 32;
    d |= (uint64_t) 1 << 46;
    return d;
}
// kind::f16, A = B = BF16, D = F32, both K-major, M = 128, N = 128
constexpr uint32_t IDESC = (1u << 4) | (OP_FMT << 7) | (OP_FMT << 10) | ((uint32_t) (BN >> 3) << 17) | ((uint32_t) (BM >> 4) << 24);

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// exp via ex2.approx (2 ulp) + fast divide: absolute error ~1e-6, far inside the 1e-3 parity tolerance
__device__ __forceinline__ float sigm(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_fast(float x) {
    const float e = __expf(2.0f * fminf(fmaxf(x, -15.0f), 15.0f));
    return 1.0f - __fdividef(2.0f, e + 1.0f);
}
__device__ __forceinline__ float selu(float x) {
    const float alpha = 1.6732632423543772848170429916717f, scale = 1.0507009873554804934193349852946f;
    return x > 0.f ? scale * x : scale * alpha * (__expf(x) - 1.0f);
}
// 8 fp32 -> 8 hi + 8 lo 16-bit operands, 16 B each
__device__ __forceinline__ void split8(const float (&v)[8], uint4 &hi, uint4 &lo) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint16_t h0 = op_bits(v[2 * i]), h1 = op_bits(v[2 * i + 1]);
        const uint16_t l0 = op_bits(v[2 * i] - op_val(h0)), l1 = op_bits(v[2 * i + 1] - op_val(h1));
        h[i] = (uint32_t) h0 | ((uint32_t) h1 << 16);
        l[i] = (uint32_t) l0 | ((uint32_t) l1 << 16);
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// ---------------------------------------------------------------- persistent variant
// One CTA per SM loops over output tiles (static round-robin).  The accumulator is double buffered in TMEM (2 x 128
// columns) and the shared-memory ring is shared by consecutive tiles, so the MMA warp starts tile i+1 while the eight
// epilogue warps are still applying the cell of tile i: the tensor pipe no longer idles during prologue / epilogue.
// Tiles are 128 x 256 here: one tcgen05.mma covers N = 256, which halves the number of MMA instructions the single
// issuing thread has to retire per FLOP (with N = 128 one thread cannot keep the tensor pipe busy; measured 52 %).
constexpr int PBN = 256;
constexpr int PSTAGES = 4;
constexpr int WTILE_ELEMS = PBN * BK;                 // 8192 bf16: weight tile image [kc][256 rows][8]
constexpr int WTILE_BYTES = WTILE_ELEMS * 2;
constexpr int PSTAGE_BYTES = 2 * TILE_BYTES + 2 * WTILE_BYTES;   // A_hi, A_lo, B_hi, B_lo = 48 KB
constexpr int PSMEM_BYTES = PSTAGES * PSTAGE_BYTES + 256;
constexpr int PTMEM_COLS = 2 * PBN;                   // double-buffered accumulator = all 512 TMEM columns
constexpr int PEPI_COLS = PBN / 2;                    // columns per epilogue warp (GRU window kernels: 8 epilogue warps)
#ifndef PB_PG_EPI_WARPS
#define PB_PG_EPI_WARPS 16
#endif
constexpr int PG_EPI_WARPS = PB_PG_EPI_WARPS;         // epilogue warps of k_tc_gemm_p: 4 TMEM lane quarters x column groups
constexpr int PG_COLS = PBN / (PG_EPI_WARPS / 4);     // columns per epilogue warp
constexpr int PG_THREADS = 64 + 32 * PG_EPI_WARPS;
constexpr uint32_t IDESC256 = (1u << 4) | (OP_FMT << 7) | (OP_FMT << 10) | ((uint32_t) (PBN >> 3) << 17) | ((uint32_t) (BM >> 4) << 24);
__device__ __forceinline__ uint64_t smem_desc_lbo(uint32_t addr, uint32_t lbo) {
    uint64_t d = 0;
    d |= (uint64_t) ((addr >> 4) & 0x3FFF);
    d |= (uint64_t) ((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t) ((128u >> 4) & 0x3FFF) << 32;
    d |= (uint64_t) 1 << 46;
    return d;
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// ---------------------------------------------------------------- e4m3 correction operands
// A weight tensor w gets a power-of-two scale 2^-E with max|w * 2^-E| in [0.5, 1) (w' = w * 2^-E).  Its fp16 images hold
// w'_hi * 2^12 and w'_lo * 2^12, its e4m3 images w'_hi and w'_lo * 2^12.  An activation a is fed as fp16 a_hi, e4m3(a) and
// e4m3(a_lo * 2^12).  Then a_hi*w_hi (fp16), e4m3(a)*e4m3(w_lo) and e4m3(a_lo)*e4m3(w_hi) all land in the fp32 accumulator
// at the same scale 2^(12-E), which the epilogue undoes exactly (Dir::acc_scale = 2^(E-12)).  The corrections carry e4m3's
// 2^-4 relative rounding on terms ~2^-12 of the product: ~2^-16 relative, below the fp16 split's own error.
//
// 8-bit operand tiles use the same K-major no-swizzle canonical layout with 16-byte core-matrix rows: for a tile of R rows
// x 32 k, element (r, k) sits at (k/16)*(R*16) + r*16 + k%16 — R*32 bytes, so the tile index arithmetic of the 16-bit
// images (TILE_ELEMS / WTILE_ELEMS elements per tile) carries over unchanged with a byte pointer.  One K32 MMA covers a
// k-tile; LBO (2048 B / 4096 B) and SBO (128 B) are the values of the 16-bit descriptors.
constexpr int TILE8_BYTES = TILE_ELEMS;               // 4 KB: 128 rows x 32 k
constexpr int WTILE8_BYTES = WTILE_ELEMS;             // 8 KB: 256 rows x 32 k
constexpr float F8_LO_SCALE = 4096.f;                 // 2^12
// Stage layout.  fp16 k-tile: A_hi | A_lo | W_hi | W_lo.  e4m3-correction k-tile: A_hi | A8_hi A8_lo | W_hi | W8_hi W8_lo
// (A8_lo / W8_hi only when the a_lo*w_hi product runs).  A_hi and W_hi sit at the same offset in both.
constexpr uint32_t ST_A_HI = 0, ST_A_LO = TILE_BYTES, ST_W_HI = 2 * TILE_BYTES, ST_W_LO = 2 * TILE_BYTES + WTILE_BYTES;
constexpr uint32_t ST_A8_HI = TILE_BYTES, ST_A8_LO = TILE_BYTES + TILE8_BYTES;
constexpr uint32_t ST_W8_HI = 2 * TILE_BYTES + WTILE_BYTES, ST_W8_LO = ST_W8_HI + WTILE8_BYTES;
static_assert(ST_A8_LO + TILE8_BYTES <= ST_W_HI && ST_W8_LO + WTILE8_BYTES <= PSTAGE_BYTES, "e4m3 stage layout");
// kind::f8f6f4, A = B = E4M3 (format 0), D = F32, both K-major, M = 128, N = 256
constexpr uint32_t IDESC256_F8 = (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t) (PBN >> 3) << 17) | ((uint32_t) (BM >> 4) << 24);

__host__ __device__ __forceinline__ uint8_t f8_bits(float v) { return (uint8_t) __nv_cvt_float_to_fp8(v, __NV_SATFINITE, __NV_E4M3); }
__device__ __forceinline__ uint32_t f8x2(float a, float b) { return (uint32_t) __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E4M3); }

__device__ __forceinline__ void tc_mma_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u) : "memory");
}

// One k-tile into stage `st`.  a8_hi != nullptr selects the e4m3-correction layout; a_lo / a8_lo == nullptr skips the a_lo*w_hi
// product (and, in e4m3 mode, the w8_hi tile it needs).
__device__ __forceinline__ void load_ktile(uint32_t st, uint32_t bar, const op_t *a_hi, const op_t *a_lo, const uint8_t *a8_hi,
                                           const uint8_t *a8_lo, const op_t *w_hi, const op_t *w_lo, const uint8_t *w8_hi,
                                           const uint8_t *w8_lo) {
    if (a8_hi) {
        mbar_expect_tx(bar, TILE_BYTES + WTILE_BYTES + TILE8_BYTES + WTILE8_BYTES + (a8_lo ? TILE8_BYTES + WTILE8_BYTES : 0u));
        bulk_g2s(st + ST_A_HI, a_hi, TILE_BYTES, bar);
        bulk_g2s(st + ST_A8_HI, a8_hi, TILE8_BYTES, bar);
        if (a8_lo) {
            bulk_g2s(st + ST_A8_LO, a8_lo, TILE8_BYTES, bar);
            bulk_g2s(st + ST_W8_HI, w8_hi, WTILE8_BYTES, bar);
        }
        bulk_g2s(st + ST_W_HI, w_hi, WTILE_BYTES, bar);
        bulk_g2s(st + ST_W8_LO, w8_lo, WTILE8_BYTES, bar);
    } else {
        mbar_expect_tx(bar, (a_lo ? 2u : 1u) * TILE_BYTES + 2u * WTILE_BYTES);
        bulk_g2s(st + ST_A_HI, a_hi, TILE_BYTES, bar);
        if (a_lo) bulk_g2s(st + ST_A_LO, a_lo, TILE_BYTES, bar);
        bulk_g2s(st + ST_W_HI, w_hi, WTILE_BYTES, bar);
        bulk_g2s(st + ST_W_LO, w_lo, WTILE_BYTES, bar);
    }
}
// The products of one k-tile in stage `st` (layout as load_ktile): fp16 a_hi*w_hi, then a_hi*w_lo (+ a_lo*w_hi) in fp16 or e4m3.
__device__ __forceinline__ void mma_ktile(uint32_t tacc, uint32_t st, bool first, bool f8, bool has_lo) {
#pragma unroll
    for (int ks = 0; ks < BK / 16; ks++) {
        const uint64_t a_hi = smem_desc_lbo(st + ST_A_HI + ks * 4096, 2048), b_hi = smem_desc_lbo(st + ST_W_HI + ks * 8192, 4096);
        tc_mma(tacc, a_hi, b_hi, IDESC256, (!first || ks > 0) ? 1u : 0u);
        if (!f8) {
            tc_mma(tacc, a_hi, smem_desc_lbo(st + ST_W_LO + ks * 8192, 4096), IDESC256, 1u);
            if (has_lo) tc_mma(tacc, smem_desc_lbo(st + ST_A_LO + ks * 4096, 2048), b_hi, IDESC256, 1u);
        }
    }
    if (f8) {
        tc_mma_f8(tacc, smem_desc_lbo(st + ST_A8_HI, 2048), smem_desc_lbo(st + ST_W8_LO, 4096), IDESC256_F8, 1u);
        if (has_lo) tc_mma_f8(tacc, smem_desc_lbo(st + ST_A8_LO, 2048), smem_desc_lbo(st + ST_W8_HI, 4096), IDESC256_F8, 1u);
    }
}

// 8 consecutive k (k0 % 8 == 0) of one row of the output operand at tile offset `tile` (elements / bytes): fp16 hi always,
// fp16 lo / e4m3 hi / e4m3 lo where the pointer is set (only the images some consumer GEMM reads are written).
__device__ __forceinline__ void put_op8(const float (&v)[8], op_t *hi, op_t *lo, uint8_t *hi8, uint8_t *lo8, int64_t tile, int k0, int r128) {
    uint32_t h[4], l[4];
    float res[8];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint16_t h0 = op_bits(v[2 * i]), h1 = op_bits(v[2 * i + 1]);
        res[2 * i] = v[2 * i] - op_val(h0);
        res[2 * i + 1] = v[2 * i + 1] - op_val(h1);
        h[i] = (uint32_t) h0 | ((uint32_t) h1 << 16);
        l[i] = (uint32_t) op_bits(res[2 * i]) | ((uint32_t) op_bits(res[2 * i + 1]) << 16);
    }
    const int64_t o = tile + (k0 >> 3) * 1024 + r128 * 8;
    *reinterpret_cast<uint4 *>(hi + o) = make_uint4(h[0], h[1], h[2], h[3]);
    if (lo) *reinterpret_cast<uint4 *>(lo + o) = make_uint4(l[0], l[1], l[2], l[3]);
    const int64_t o8 = tile + (k0 >> 4) * 2048 + r128 * 16 + (k0 & 15);
    if (hi8)
        *reinterpret_cast<uint2 *>(hi8 + o8) = make_uint2(f8x2(v[0], v[1]) | (f8x2(v[2], v[3]) << 16), f8x2(v[4], v[5]) | (f8x2(v[6], v[7]) << 16));
    if (lo8) {
        float s[8];
#pragma unroll
        for (int i = 0; i < 8; i++) s[i] = res[i] * F8_LO_SCALE;
        *reinterpret_cast<uint2 *>(lo8 + o8) = make_uint2(f8x2(s[0], s[1]) | (f8x2(s[2], s[3]) << 16), f8x2(s[4], s[5]) | (f8x2(s[6], s[7]) << 16));
    }
}

template <int EPI>
__global__ void __launch_bounds__(PG_THREADS, 1) k_tc_gemm_p(Args G, int n_mt, int n_nt /* 256-column tiles */, int n_dir) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + PSTAGES * PSTAGE_BYTES);
    const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + PSTAGES);
    const uint32_t bar_accf = smem_u32(bars + 2 * PSTAGES), bar_acce = smem_u32(bars + 2 * PSTAGES + 2);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * PSTAGES + 4);
    const uint32_t smem_base = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tiles = n_mt * n_nt * n_dir;

    if (threadIdx.x == 0) {
        for (int s = 0; s < PSTAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int b = 0; b < 2; b++) { mbar_init(bar_accf + 8 * b, 1); mbar_init(bar_acce + 8 * b, PG_EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t) PTMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // tile -> (dir, mt, nt): nt fastest so that CTAs running together share the A row tile
    auto decode = [&](int tile, int &dir, int &mt, int &nt) {
        nt = tile % n_nt;
        const int r = tile / n_nt;
        mt = r % n_mt;
        dir = r / n_mt;
    };

    if (warp == 0) {
        if (lane == 0) {
            uint32_t g = 0;                                   // running k-tile counter across tiles
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                int dir, mt, nt;
                decode(tile, dir, mt, nt);
                const Dir &D = G.d[dir];
                const int nkt0 = D.seg[0].nkt, nkt = nkt0 + D.seg[1].nkt;
                for (int kt = 0; kt < nkt; kt++, g++) {
                    const uint32_t s = g % PSTAGES, ph = (g / PSTAGES) & 1u;
                    mbar_wait(bar_empty + 8 * s, ph ^ 1u);
                    const Seg &S = (kt < nkt0) ? D.seg[0] : D.seg[1];
                    const int64_t off = (int64_t) mt * S.mt_stride + (int64_t) ((kt < nkt0) ? kt : kt - nkt0) * TILE_ELEMS;
                    const int64_t woff = ((int64_t) nt * D.w_nkt + kt) * WTILE_ELEMS;
                    load_ktile(smem_base + s * PSTAGE_BYTES, bar_full + 8 * s, S.hi + off, S.lo ? S.lo + off : nullptr,
                               S.hi8 ? S.hi8 + off : nullptr, S.lo8 ? S.lo8 + off : nullptr, D.w_hi + woff, D.w_lo + woff,
                               D.w8_hi ? D.w8_hi + woff : nullptr, D.w8_lo ? D.w8_lo + woff : nullptr);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t g = 0, it = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, it++) {
                int dir, mt, nt;
                decode(tile, dir, mt, nt);
                const Dir &D = G.d[dir];
                const int nkt0 = D.seg[0].nkt, nkt = nkt0 + D.seg[1].nkt;
                const uint32_t buf = it & 1u, use = it >> 1;
                mbar_wait(bar_acce + 8 * buf, (use & 1u) ^ 1u);        // epilogue has drained this accumulator buffer
                tc_fence_after();
                const uint32_t tacc = tmem_base + buf * PBN;
                for (int kt = 0; kt < nkt; kt++, g++) {
                    const uint32_t s = g % PSTAGES, ph = (g / PSTAGES) & 1u;
                    mbar_wait(bar_full + 8 * s, ph);
                    tc_fence_after();
                    const Seg &S = (kt < nkt0) ? D.seg[0] : D.seg[1];
                    const bool f8 = S.hi8 != nullptr;
                    mma_ktile(tacc, smem_base + s * PSTAGE_BYTES, kt == 0, f8, (f8 ? (const void *) S.lo8 : (const void *) S.lo) != nullptr);
                    tc_commit(bar_empty + 8 * s);
                }
                tc_commit(bar_accf + 8 * buf);
            }
        }
    } else {
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;
        const int r128 = q * 32 + lane;
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, it++) {
            int dir, mt, nt;
            decode(tile, dir, mt, nt);
            const Dir &D = G.d[dir];
            const uint32_t buf = it & 1u, use = it >> 1;
            const int row = mt * BM + r128;
            const bool valid = row < G.M;
            float st[PG_COLS / 4];
            const int ubase = nt * (PBN / 4) + half * (PG_COLS / 4);
            if (EPI == EPI_LSTM) {
#pragma unroll
                for (int u = 0; u < PG_COLS / 4; u++) st[u] = valid ? D.c[(int64_t) (ubase + u) * G.c_ld + row] : 0.f;
            } else if (EPI == EPI_GRU) {
#pragma unroll
                for (int u8 = 0; u8 < PG_COLS / 32; u8++) {
                    uint4 h = make_uint4(0, 0, 0, 0), l = make_uint4(0, 0, 0, 0);
                    if (valid && D.hp_hi) {
                        const int j0 = ubase + u8 * 8;
                        const int64_t o = (int64_t) mt * D.hp_mt_stride + (int64_t) (j0 >> 5) * TILE_ELEMS + ((j0 & 31) >> 3) * 1024 + r128 * 8;
                        h = *reinterpret_cast<const uint4 *>(D.hp_hi + o);
                        l = *reinterpret_cast<const uint4 *>(D.hp_lo + o);
                    }
                    const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
                    for (int e = 0; e < 8; e++)
                        st[u8 * 8 + e] = op_val(hw[e >> 1] >> (16 * (e & 1))) + op_val(lw[e >> 1] >> (16 * (e & 1)));
                }
            }
            mbar_wait(bar_accf + 8 * buf, use & 1u);
            tc_fence_after();
#pragma unroll
            for (int cl = 0; cl < PG_COLS / 32; cl++) {
                const int cc = half * (PG_COLS / 32) + cl;
                const int col0 = nt * PBN + cc * 32;
                uint32_t acc[32];
                tmem_ld32(tmem_base + buf * PBN + ((uint32_t) (q * 32) << 16) + (uint32_t) (cc * 32), acc);
                if (cl == PG_COLS / 32 - 1) {
                    // last read of this accumulator buffer by this warp: hand it back to the MMA warp
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_acce + 8 * buf);
                }
                if (EPI == EPI_BIAS || EPI == EPI_SELU) {
#pragma unroll
                    for (int g8 = 0; g8 < 4; g8++) {
                        float v[8];
#pragma unroll
                        for (int i = 0; i < 8; i++) {
                            const float x = __uint_as_float(acc[g8 * 8 + i]) * D.acc_scale + __ldg(D.bias + col0 + g8 * 8 + i);
                            v[i] = (EPI == EPI_SELU) ? selu(x) : x;
                        }
                        if (valid) {
                            if (D.y_hi)
                                put_op8(v, D.y_hi, D.y_lo, D.y_hi8, D.y_lo8, (int64_t) mt * D.y_mt_stride + (int64_t) (D.y_kt0 + col0 / 32) * TILE_ELEMS,
                                        g8 * 8, r128);
                            if (D.y_f32) {
                                float4 *dst = reinterpret_cast<float4 *>(D.y_f32 + (int64_t) row * D.ldy + col0 + g8 * 8);
                                dst[0] = make_float4(v[0], v[1], v[2], v[3]);
                                dst[1] = make_float4(v[4], v[5], v[6], v[7]);
                            }
                        }
                    }
                } else {
                    const int j0 = col0 >> 2;
                    float hn[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const float4 bz = __ldg(reinterpret_cast<const float4 *>(D.bias + col0 + 4 * u));
                        const float sc = D.acc_scale;
                        const float v0 = __uint_as_float(acc[4 * u + 0]) * sc + bz.x, v1 = __uint_as_float(acc[4 * u + 1]) * sc + bz.y;
                        const float v2 = __uint_as_float(acc[4 * u + 2]) * sc + bz.z, v3 = __uint_as_float(acc[4 * u + 3]) * sc + bz.w;
                        if (EPI == EPI_LSTM) {
                            const float ig = sigm(v0), fg = sigm(v1), gg = tanh_fast(v2), og = sigm(v3);
                            const float cn = fg * st[cl * 8 + u] + ig * gg;
                            st[cl * 8 + u] = cn;
                            hn[u] = og * tanh_fast(cn);
                        } else {
                            const float r = sigm(v0), z = sigm(v1);
                            const float n = tanh_fast(v2 + r * v3);
                            hn[u] = (1.0f - z) * n + z * st[cl * 8 + u];
                        }
                    }
                    if (valid) {
                        put_op8(hn, D.y_hi, D.y_lo, D.y_hi8, D.y_lo8, (int64_t) mt * D.y_mt_stride + (int64_t) (D.y_kt0 + (j0 >> 5)) * TILE_ELEMS,
                                j0 & 31, r128);
                        if (D.y_f32) {
                            float4 *dst = reinterpret_cast<float4 *>(D.y_f32 + (int64_t) row * D.ldy + j0);
                            dst[0] = make_float4(hn[0], hn[1], hn[2], hn[3]);
                            dst[1] = make_float4(hn[4], hn[5], hn[6], hn[7]);
                        }
                    }
                }
            }
            if (EPI == EPI_LSTM && valid) {
#pragma unroll
                for (int u = 0; u < PG_COLS / 4; u++) D.c[(int64_t) (ubase + u) * G.c_ld + row] = st[u];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t) PTMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------- persistent LSTM layer kernel (variant)
// All T time steps of one bidirectional LSTM layer in ONE launch.  CTA b owns (direction, 128-candidate row tile) for the
// whole sequence and computes all four 256-column gate tiles of every step itself, so the recurrence never leaves the
// CTA: the epilogue writes h_t as bf16 hi/lo operand tiles into the layer's output sequence, arrives on a CTA-local
// mbarrier, and the producer thread loads those tiles back as the h-part of step t+1 (generic -> async proxy fence in
// between).  The x-part of step t+1 (1 k-tile for the encoder layer, 16 for the decoder layer) does not depend on h_t and
// is streamed / multiplied while the last epilogue of step t drains; the TMEM accumulator stays double buffered across
// tiles and steps.  One chunk of 9,472 candidates = 74 row tiles x 2 directions = 148 CTAs = one per SM; 33 x fewer
// launches, prologues and tails than the per-step kernel above (kept as the cross-check path).
struct LstmLayer {
    const op_t *x_hi, *x_lo;           // input sequence operand: tile (mt, t, kt) at mt * x_mt_stride + (t * x_nkt + kt) * TILE_ELEMS
    const uint8_t *x_hi8, *x_lo8;      // its e4m3 images (same tile offsets, bytes)
    int64_t x_mt_stride;
    int x_nkt;
    const op_t *w_hi[2], *w_lo[2];     // per direction: [4 n-tiles][x_nkt + 8][WTILE_ELEMS]
    const uint8_t *w8_hi[2], *w8_lo[2];
    float acc_scale[2];                // accumulator -> gate pre-activation (2^(E-12) of the direction's weight scale)
    const float *bias[2];
    float *c[2];                                // cell state per direction [256][c_ld], zero initialised
    op_t *y_hi, *y_lo;                 // output sequence operand [mt][T][16] tiles; (time tt, direction d) -> k-tiles tt * 16 + d * 8 ...
    uint8_t *y_hi8, *y_lo8;            // its e4m3 images; y_lo / y_hi8 / y_lo8 == nullptr: not written (no consumer reads it)
    int64_t y_mt_stride;
    float *y_f32;                               // optional fp32 copy [row][T][512]
    int64_t ldy;
    int M, n_mt, T;
    int64_t c_ld;
    int lo_x, lo_h;                             // 1: the a_lo x w_hi product of the x-part / h-part is executed (0: two products)
    int f8_x, f8_h;                             // 1: the corrections of the x-part / h-part run in e4m3
};

__global__ void __launch_bounds__(PG_THREADS, 1) k_lstm_layer(LstmLayer G) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + PSTAGES * PSTAGE_BYTES);
    const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + PSTAGES);
    const uint32_t bar_accf = smem_u32(bars + 2 * PSTAGES), bar_acce = smem_u32(bars + 2 * PSTAGES + 2);
    const uint32_t bar_h = smem_u32(bars + 2 * PSTAGES + 4);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * PSTAGES + 5);
    const uint32_t smem_base = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int dir = blockIdx.x / G.n_mt, mt = blockIdx.x % G.n_mt;
    const int w_nkt = G.x_nkt + 8;

    if (threadIdx.x == 0) {
        for (int s = 0; s < PSTAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int b = 0; b < 2; b++) { mbar_init(bar_accf + 8 * b, 1); mbar_init(bar_acce + 8 * b, PG_EPI_WARPS); }
        mbar_init(bar_h, PG_EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t) PTMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t g = 0;
            for (int t = 0; t < G.T; t++) {
                const int tt = dir ? G.T - 1 - t : t, tp = dir ? tt + 1 : tt - 1;
                const int nkt = G.x_nkt + (t > 0 ? 8 : 0);
                for (int nt = 0; nt < 4; nt++) {
                    for (int kt = 0; kt < nkt; kt++, g++) {
                        const uint32_t s = g % PSTAGES, ph = (g / PSTAGES) & 1u;
                        mbar_wait(bar_empty + 8 * s, ph ^ 1u);
                        const op_t *a_hi, *a_lo = nullptr;
                        const uint8_t *a8_hi = nullptr, *a8_lo = nullptr;
                        if (kt < G.x_nkt) {
                            const int64_t off = (int64_t) mt * G.x_mt_stride + ((int64_t) tt * G.x_nkt + kt) * TILE_ELEMS;
                            a_hi = G.x_hi + off;
                            if (G.f8_x) { a8_hi = G.x_hi8 + off; if (G.lo_x) a8_lo = G.x_lo8 + off; }
                            else if (G.lo_x) a_lo = G.x_lo + off;
                        } else {
                            const int kk = kt - G.x_nkt;
                            if (kk == 0 && nt == 0) {
                                // every epilogue warp has written its part of h_{t-1}: make it visible to the bulk-copy engine
                                mbar_wait(bar_h, (uint32_t) (t - 1) & 1u);
                                asm volatile("fence.proxy.async;" ::: "memory");
                            }
                            const int64_t off = (int64_t) mt * G.y_mt_stride + ((int64_t) tp * 16 + dir * 8 + kk) * TILE_ELEMS;
                            a_hi = G.y_hi + off;
                            if (G.f8_h) { a8_hi = G.y_hi8 + off; if (G.lo_h) a8_lo = G.y_lo8 + off; }
                            else if (G.lo_h) a_lo = G.y_lo + off;
                        }
                        const int64_t woff = ((int64_t) nt * w_nkt + kt) * WTILE_ELEMS;
                        load_ktile(smem_base + s * PSTAGE_BYTES, bar_full + 8 * s, a_hi, a_lo, a8_hi, a8_lo, G.w_hi[dir] + woff,
                                   G.w_lo[dir] + woff, G.w8_hi[dir] ? G.w8_hi[dir] + woff : nullptr, G.w8_lo[dir] ? G.w8_lo[dir] + woff : nullptr);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t g = 0, it = 0;
            for (int t = 0; t < G.T; t++) {
                const int nkt = G.x_nkt + (t > 0 ? 8 : 0);
                for (int nt = 0; nt < 4; nt++, it++) {
                    const uint32_t buf = it & 1u, use = it >> 1;
                    mbar_wait(bar_acce + 8 * buf, (use & 1u) ^ 1u);
                    tc_fence_after();
                    const uint32_t tacc = tmem_base + buf * PBN;
                    for (int kt = 0; kt < nkt; kt++, g++) {
                        const uint32_t s = g % PSTAGES, ph = (g / PSTAGES) & 1u;
                        mbar_wait(bar_full + 8 * s, ph);
                        tc_fence_after();
                        const bool xpart = kt < G.x_nkt;
                        mma_ktile(tacc, smem_base + s * PSTAGE_BYTES, kt == 0, (xpart ? G.f8_x : G.f8_h) != 0, (xpart ? G.lo_x : G.lo_h) != 0);
                        tc_commit(bar_empty + 8 * s);
                    }
                    tc_commit(bar_accf + 8 * buf);
                }
            }
        }
    } else {
        const int q = warp & 3;
        const int grp = (warp - 2) >> 2;                        // column group of this warp inside a 256-column tile
        const int r128 = q * 32 + lane;
        const int row = mt * BM + r128;
        const bool valid = row < G.M;
        float *cst = G.c[dir];
        const float *bias = G.bias[dir];
        const float sc = G.acc_scale[dir];
        uint32_t it = 0;
        for (int t = 0; t < G.T; t++) {
            const int tt = dir ? G.T - 1 - t : t;
            const int y_kt0 = tt * 16 + dir * 8;
            for (int nt = 0; nt < 4; nt++, it++) {
                const uint32_t buf = it & 1u, use = it >> 1;
                float st[PG_COLS / 4];
                const int ubase = nt * (PBN / 4) + grp * (PG_COLS / 4);
#pragma unroll
                for (int u = 0; u < PG_COLS / 4; u++) st[u] = valid ? cst[(int64_t) (ubase + u) * G.c_ld + row] : 0.f;
                mbar_wait(bar_accf + 8 * buf, use & 1u);
                tc_fence_after();
#pragma unroll
                for (int cl = 0; cl < PG_COLS / 32; cl++) {
                    const int cc = grp * (PG_COLS / 32) + cl;
                    const int col0 = nt * PBN + cc * 32;
                    uint32_t acc[32];
                    tmem_ld32(tmem_base + buf * PBN + ((uint32_t) (q * 32) << 16) + (uint32_t) (cc * 32), acc);
                    if (cl == PG_COLS / 32 - 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(bar_acce + 8 * buf);
                    }
                    const int j0 = col0 >> 2;
                    float hn[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const float4 bz = __ldg(reinterpret_cast<const float4 *>(bias + col0 + 4 * u));
                        const float v0 = __uint_as_float(acc[4 * u + 0]) * sc + bz.x, v1 = __uint_as_float(acc[4 * u + 1]) * sc + bz.y;
                        const float v2 = __uint_as_float(acc[4 * u + 2]) * sc + bz.z, v3 = __uint_as_float(acc[4 * u + 3]) * sc + bz.w;
                        const float ig = sigm(v0), fg = sigm(v1), gg = tanh_fast(v2), og = sigm(v3);
                        const float cn = fg * st[cl * 8 + u] + ig * gg;
                        st[cl * 8 + u] = cn;
                        hn[u] = og * tanh_fast(cn);
                    }
                    if (valid) {
                        put_op8(hn, G.y_hi, G.y_lo, G.y_hi8, G.y_lo8, (int64_t) mt * G.y_mt_stride + (int64_t) (y_kt0 + (j0 >> 5)) * TILE_ELEMS,
                                j0 & 31, r128);
                        if (G.y_f32) {
                            float4 *dst = reinterpret_cast<float4 *>(G.y_f32 + (int64_t) row * G.ldy + (int64_t) tt * 512 + dir * 256 + j0);
                            dst[0] = make_float4(hn[0], hn[1], hn[2], hn[3]);
                            dst[1] = make_float4(hn[4], hn[5], hn[6], hn[7]);
                        }
                    }
                }
                if (valid) {
#pragma unroll
                    for (int u = 0; u < PG_COLS / 4; u++) cst[(int64_t) (ubase + u) * G.c_ld + row] = st[u];
                }
                if (nt == 3) {
                    // h_t of this warp's rows / columns is complete (all four gate tiles): publish it to the producer thread
                    __threadfence();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_h);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t) PTMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------- GRU window layers (polish)
// All 100 time steps of one bidirectional GRU layer of one window in ONE launch (k_gru_layer below; k_gru_cluster is the A/B
// fallback that splits the hidden units over a 2-CTA cluster).  The first persistent version, k_gru_window (sibling CTAs
// exchanging h through HBM flags under a cooperative launch), was removed in round 2: superseded twice.
struct GruWin {
    const op_t *x_hi, *x_lo;      // input sequence operand [mt][100][x_kt] tiles (x_lo == nullptr: exact input)
    int x_kt;
    const op_t *h0_hi[2], *h0_lo[2];   // initial state tiles per direction (4 k-tiles per row tile)
    int64_t h0_mt_stride;
    const op_t *w_hi[2], *w_lo[2];     // per direction: [nt(2)][x_kt + 4][WTILE_ELEMS]
    const float *bias[2];
    op_t *y_hi, *y_lo;            // output sequence operand [mt][100][8] tiles
    int *flags;                            // unused (kept for layout stability of the host code)
    int M, n_mt, T;
    int lo_x, lo_h;                        // k_gru_layer: 1 = execute the a_lo x w_hi product of the x-part / h-part
};

// ---------------------------------------------------------------- cluster-resident GRU window kernel (polish)
// Same work split as k_gru_window, but the two CTAs that own the two halves of a (direction, row tile) form a thread-block
// CLUSTER and exchange h_t through distributed shared memory instead of HBM: the epilogue writes its 64 units of h_t (bf16
// hi/lo operand tiles) into the local H buffer, one thread pushes them to the sibling's H buffer with
// cp.async.bulk.shared::cluster (completing on the sibling's mbarrier), and the MMA warp of each CTA feeds the h part of
// the next step straight from its H buffer.  The per-step critical path loses the store -> fence -> flag -> poll -> L2
// round trip; there is no cross-cluster dependency, so any batch size runs (no cooperative launch).
constexpr int CSTAGES = 2;
constexpr int HBUF_BYTES = 4 * 2 * TILE_BYTES;                  // 4 k-tiles x (hi, lo) = 64 KB
constexpr int CSMEM_BYTES = 2 * HBUF_BYTES + CSTAGES * PSTAGE_BYTES + 256;

__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1) k_gru_cluster(GruWin G) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t *ring = smem + 2 * HBUF_BYTES;
    uint64_t *bars = reinterpret_cast<uint64_t *>(ring + CSTAGES * PSTAGE_BYTES);
    const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + CSTAGES);
    const uint32_t bar_accf = smem_u32(bars + 2 * CSTAGES), bar_acce = smem_u32(bars + 2 * CSTAGES + 2);
    const uint32_t bar_h = smem_u32(bars + 2 * CSTAGES + 4);               // h_ready[2]
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * CSTAGES + 6);
    const uint32_t hbuf = smem_u32(smem), ring_base = smem_u32(ring);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nt = blockIdx.x & 1, pair = blockIdx.x >> 1;                // nt == rank in the cluster
    const int mt = pair % G.n_mt, dir = pair / G.n_mt;
    const int nkt = G.x_kt + 4;
    const int64_t seq_stride = (int64_t) G.T * 8 * TILE_ELEMS;

    if (threadIdx.x == 0) {
        for (int s = 0; s < CSTAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int b = 0; b < 2; b++) { mbar_init(bar_accf + 8 * b, 1); mbar_init(bar_acce + 8 * b, 8); mbar_init(bar_h + 8 * b, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t) PTMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                      // the sibling's barriers exist before anything is sent to them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // initial state -> H[1] (the "t-1" buffer of step 0)
            mbar_expect_tx(bar_h + 8, 8u * TILE_BYTES);
            for (int kk = 0; kk < 4; kk++) {
                const int64_t off = (int64_t) mt * G.h0_mt_stride + (int64_t) kk * TILE_ELEMS;
                bulk_g2s(hbuf + HBUF_BYTES + kk * 2 * TILE_BYTES, G.h0_hi[dir] + off, TILE_BYTES, bar_h + 8);
                bulk_g2s(hbuf + HBUF_BYTES + kk * 2 * TILE_BYTES + TILE_BYTES, G.h0_lo[dir] + off, TILE_BYTES, bar_h + 8);
            }
            uint32_t g = 0;
            for (int t = 0; t < G.T; t++) {
                const int tt = dir == 0 ? t : G.T - 1 - t;
                for (int kt = 0; kt < nkt; kt++, g++) {
                    const uint32_t s = g % CSTAGES, ph = (g / CSTAGES) & 1u;
                    mbar_wait(bar_empty + 8 * s, ph ^ 1u);
                    const uint32_t st = ring_base + s * PSTAGE_BYTES;
                    const int64_t woff = ((int64_t) nt * nkt + kt) * WTILE_ELEMS;
                    if (kt < G.x_kt) {
                        const int64_t off = ((int64_t) (mt * G.T + tt) * G.x_kt + kt) * TILE_ELEMS;
                        mbar_expect_tx(bar_full + 8 * s, (G.x_lo ? 2u : 1u) * TILE_BYTES + 2u * WTILE_BYTES);
                        bulk_g2s(st, G.x_hi + off, TILE_BYTES, bar_full + 8 * s);
                        if (G.x_lo) bulk_g2s(st + TILE_BYTES, G.x_lo + off, TILE_BYTES, bar_full + 8 * s);
                    } else {
                        mbar_expect_tx(bar_full + 8 * s, 2u * WTILE_BYTES);      // A comes from the resident H buffer
                    }
                    bulk_g2s(st + 2 * TILE_BYTES, G.w_hi[dir] + woff, WTILE_BYTES, bar_full + 8 * s);
                    bulk_g2s(st + 2 * TILE_BYTES + WTILE_BYTES, G.w_lo[dir] + woff, WTILE_BYTES, bar_full + 8 * s);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t g = 0;
            for (int t = 0; t < G.T; t++) {
                const uint32_t buf = (uint32_t) t & 1u, use = (uint32_t) t >> 1;
                mbar_wait(bar_acce + 8 * buf, (use & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t tacc = tmem_base + buf * PBN;
                const uint32_t hsrc = hbuf + (((uint32_t) (t + 1)) & 1u) * HBUF_BYTES;     // H[(t-1)&1]
                for (int kt = 0; kt < nkt; kt++, g++) {
                    const uint32_t s = g % CSTAGES, ph = (g / CSTAGES) & 1u;
                    mbar_wait(bar_full + 8 * s, ph);
                    const bool xpart = kt < G.x_kt;
                    if (kt == G.x_kt) mbar_wait(bar_h + 8 * (((uint32_t) (t + 1)) & 1u), ((uint32_t) t >> 1) & 1u);   // h_{t-1} complete
                    tc_fence_after();
                    const bool has_lo = !xpart || (G.x_lo != nullptr);
                    const uint32_t st = ring_base + s * PSTAGE_BYTES;
                    const uint32_t a_base = xpart ? st : hsrc + (uint32_t) (kt - G.x_kt) * 2 * TILE_BYTES;
#pragma unroll
                    for (int ks = 0; ks < BK / 16; ks++) {
                        const uint64_t a_hi = smem_desc_lbo(a_base + ks * 4096, 2048), a_lo = smem_desc_lbo(a_base + TILE_BYTES + ks * 4096, 2048);
                        const uint64_t b_hi = smem_desc_lbo(st + 2 * TILE_BYTES + ks * 8192, 4096);
                        const uint64_t b_lo = smem_desc_lbo(st + 2 * TILE_BYTES + WTILE_BYTES + ks * 8192, 4096);
                        tc_mma(tacc, a_hi, b_hi, IDESC256, (kt > 0 || ks > 0) ? 1u : 0u);
                        tc_mma(tacc, a_hi, b_lo, IDESC256, 1u);
                        if (has_lo) tc_mma(tacc, a_lo, b_hi, IDESC256, 1u);
                    }
                    tc_commit(bar_empty + 8 * s);
                }
                tc_commit(bar_accf + 8 * buf);
            }
        }
    } else {
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;
        const int r128 = q * 32 + lane;
        const int row = mt * BM + r128;
        const bool valid = row < G.M;
        const int ubase = nt * (PBN / 4) + half * (PEPI_COLS / 4);
        const float *bias = G.bias[dir];
        float hp[PEPI_COLS / 4];
#pragma unroll
        for (int u8 = 0; u8 < PEPI_COLS / 32; u8++) {
            uint4 h = make_uint4(0, 0, 0, 0), l = make_uint4(0, 0, 0, 0);
            if (valid) {
                const int j0 = ubase + u8 * 8;
                const int64_t o = (int64_t) mt * G.h0_mt_stride + (int64_t) (j0 >> 5) * TILE_ELEMS + ((j0 & 31) >> 3) * 1024 + r128 * 8;
                h = *reinterpret_cast<const uint4 *>(G.h0_hi[dir] + o);
                l = *reinterpret_cast<const uint4 *>(G.h0_lo[dir] + o);
            }
            const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
            for (int e = 0; e < 8; e++)
                hp[u8 * 8 + e] = op_val(hw[e >> 1] >> (16 * (e & 1))) + op_val(lw[e >> 1] >> (16 * (e & 1)));
        }
        const uint32_t peer = (uint32_t) (nt ^ 1);
        for (int t = 0; t < G.T; t++) {
            const int tt = dir == 0 ? t : G.T - 1 - t;
            const uint32_t buf = (uint32_t) t & 1u, use = (uint32_t) t >> 1;
            uint8_t *hdst = smem + buf * HBUF_BYTES;                                   // H[t&1]
            mbar_wait(bar_accf + 8 * buf, use & 1u);
            tc_fence_after();
#pragma unroll
            for (int cl = 0; cl < PEPI_COLS / 32; cl++) {
                const int cc = half * (PEPI_COLS / 32) + cl;
                const int col0 = nt * PBN + cc * 32;
                uint32_t acc[32];
                tmem_ld32(tmem_base + buf * PBN + ((uint32_t) (q * 32) << 16) + (uint32_t) (cc * 32), acc);
                if (cl == PEPI_COLS / 32 - 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_acce + 8 * buf);
                }
                const int j0 = col0 >> 2;
                float hn[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const float4 bz = __ldg(reinterpret_cast<const float4 *>(bias + col0 + 4 * u));
                    const float v0 = __uint_as_float(acc[4 * u + 0]) + bz.x, v1 = __uint_as_float(acc[4 * u + 1]) + bz.y;
                    const float v2 = __uint_as_float(acc[4 * u + 2]) + bz.z, v3 = __uint_as_float(acc[4 * u + 3]) + bz.w;
                    const float r = sigm(v0), z = sigm(v1);
                    const float n = tanh_fast(v2 + r * v3);
                    hn[u] = (1.0f - z) * n + z * hp[cl * 8 + u];
                    hp[cl * 8 + u] = hn[u];
                }
                uint4 hi, lo;
                split8(hn, hi, lo);
                // local H buffer (rows beyond M carry zeros-derived values; harmless, never stored to HBM)
                const uint32_t so = (uint32_t) (j0 >> 5) * 2 * TILE_BYTES + (uint32_t) (((j0 & 31) >> 3) * 1024 + r128 * 8) * 2;
                *reinterpret_cast<uint4 *>(hdst + so) = hi;
                *reinterpret_cast<uint4 *>(hdst + so + TILE_BYTES) = lo;
                if (valid) {
                    const int64_t o = (int64_t) mt * seq_stride + ((int64_t) tt * 8 + dir * 4 + (j0 >> 5)) * TILE_ELEMS + ((j0 & 31) >> 3) * 1024 + r128 * 8;
                    *reinterpret_cast<uint4 *>(G.y_hi + o) = hi;
                    *reinterpret_cast<uint4 *>(G.y_lo + o) = lo;
                }
            }
            if (t + 1 < G.T) {
                // my two k-tiles of h_t are in the local H buffer: make them visible to the async proxy, then one thread
                // announces them locally and pushes them into the sibling's H buffer (completing on ITS barrier)
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("bar.sync 1, 256;" ::: "memory");
                if (threadIdx.x == 64) {
                    mbar_expect_tx(bar_h + 8 * buf, 4u * TILE_BYTES);                // the sibling's two k-tiles (hi, lo) will land here
                    const uint32_t rbar = mapa_u32(bar_h + 8 * buf, peer);
#pragma unroll
                    for (int k2 = 0; k2 < 2; k2++) {
                        const uint32_t off = (uint32_t) buf * HBUF_BYTES + (uint32_t) (2 * nt + k2) * 2 * TILE_BYTES;
                        const uint32_t rdst = mapa_u32(hbuf + off, peer);
                        asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                     ::"r"(rdst), "r"(hbuf + off), "r"(2u * TILE_BYTES), "r"(rbar) : "memory");
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                      // nobody exits while the sibling may still write into its shared memory
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t) PTMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------- persistent GRU layer kernel, one CTA per (direction, row tile)
// Same ownership as k_lstm_layer: the CTA computes both 256-column gate tiles (128 hidden units x {r, z, n_x, n_h}) of every
// step, so h never has to be exchanged with a sibling CTA (k_gru_cluster / k_gru_window split the hidden units over a CTA
// pair).  h_t goes out as operand tiles of the layer's output sequence and comes back through the bulk-copy ring as the
// h-part of step t+1; the previous hidden values of the cell update are re-read from those tiles (L2).  Step 0 takes h0.
__global__ void __launch_bounds__(PG_THREADS, 1) k_gru_layer(GruWin G) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + PSTAGES * PSTAGE_BYTES);
    const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + PSTAGES);
    const uint32_t bar_accf = smem_u32(bars + 2 * PSTAGES), bar_acce = smem_u32(bars + 2 * PSTAGES + 2);
    const uint32_t bar_h = smem_u32(bars + 2 * PSTAGES + 4);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * PSTAGES + 5);
    const uint32_t smem_base = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int dir = blockIdx.x / G.n_mt, mt = blockIdx.x % G.n_mt;
    const int nkt = G.x_kt + 4;
    const int64_t seq_stride = (int64_t) G.T * 8 * TILE_ELEMS;

    if (threadIdx.x == 0) {
        for (int s = 0; s < PSTAGES; s++) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
        for (int b = 0; b < 2; b++) { mbar_init(bar_accf + 8 * b, 1); mbar_init(bar_acce + 8 * b, PG_EPI_WARPS); }
        mbar_init(bar_h, PG_EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t) PTMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t g = 0;
            for (int t = 0; t < G.T; t++) {
                const int tt = dir ? G.T - 1 - t : t, tp = dir ? tt + 1 : tt - 1;
                for (int nt = 0; nt < 2; nt++) {
                    for (int kt = 0; kt < nkt; kt++, g++) {
                        const uint32_t s = g % PSTAGES, ph = (g / PSTAGES) & 1u;
                        mbar_wait(bar_empty + 8 * s, ph ^ 1u);
                        const op_t *a_hi, *a_lo;
                        if (kt < G.x_kt) {
                            const int64_t off = ((int64_t) (mt * G.T + tt) * G.x_kt + kt) * TILE_ELEMS;
                            a_hi = G.x_hi + off; a_lo = (G.x_lo && G.lo_x) ? G.x_lo + off : nullptr;
                        } else {
                            const int kk = kt - G.x_kt;
                            if (t == 0) {
                                const int64_t off = (int64_t) mt * G.h0_mt_stride + (int64_t) kk * TILE_ELEMS;
                                a_hi = G.h0_hi[dir] + off; a_lo = G.lo_h ? G.h0_lo[dir] + off : nullptr;
                            } else {
                                if (kk == 0 && nt == 0) {
                                    mbar_wait(bar_h, (uint32_t) (t - 1) & 1u);      // every epilogue warp has written its part of h_{t-1}
                                    asm volatile("fence.proxy.async;" ::: "memory");
                                }
                                const int64_t off = (int64_t) mt * seq_stride + ((int64_t) tp * 8 + dir * 4 + kk) * TILE_ELEMS;
                                a_hi = G.y_hi + off; a_lo = G.lo_h ? G.y_lo + off : nullptr;
                            }
                        }
                        const uint32_t st = smem_base + s * PSTAGE_BYTES;
                        mbar_expect_tx(bar_full + 8 * s, (a_lo ? 2u : 1u) * TILE_BYTES + 2u * WTILE_BYTES);
                        bulk_g2s(st, a_hi, TILE_BYTES, bar_full + 8 * s);
                        if (a_lo) bulk_g2s(st + TILE_BYTES, a_lo, TILE_BYTES, bar_full + 8 * s);
                        const int64_t woff = ((int64_t) nt * nkt + kt) * WTILE_ELEMS;
                        bulk_g2s(st + 2 * TILE_BYTES, G.w_hi[dir] + woff, WTILE_BYTES, bar_full + 8 * s);
                        bulk_g2s(st + 2 * TILE_BYTES + WTILE_BYTES, G.w_lo[dir] + woff, WTILE_BYTES, bar_full + 8 * s);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            uint32_t g = 0, it = 0;
            for (int t = 0; t < G.T; t++) {
                for (int nt = 0; nt < 2; nt++, it++) {
                    const uint32_t buf = it & 1u, use = it >> 1;
                    mbar_wait(bar_acce + 8 * buf, (use & 1u) ^ 1u);
                    tc_fence_after();
                    const uint32_t tacc = tmem_base + buf * PBN;
                    for (int kt = 0; kt < nkt; kt++, g++) {
                        const uint32_t s = g % PSTAGES, ph = (g / PSTAGES) & 1u;
                        mbar_wait(bar_full + 8 * s, ph);
                        tc_fence_after();
                        const bool has_lo = kt >= G.x_kt ? (G.lo_h != 0) : (G.x_lo != nullptr && G.lo_x != 0);
                        const uint32_t st = smem_base + s * PSTAGE_BYTES;
#pragma unroll
                        for (int ks = 0; ks < BK / 16; ks++) {
                            const uint64_t a_hi = smem_desc_lbo(st + ks * 4096, 2048), a_lo = smem_desc_lbo(st + TILE_BYTES + ks * 4096, 2048);
                            const uint64_t b_hi = smem_desc_lbo(st + 2 * TILE_BYTES + ks * 8192, 4096);
                            const uint64_t b_lo = smem_desc_lbo(st + 2 * TILE_BYTES + WTILE_BYTES + ks * 8192, 4096);
                            tc_mma(tacc, a_hi, b_hi, IDESC256, (kt > 0 || ks > 0) ? 1u : 0u);
                            tc_mma(tacc, a_hi, b_lo, IDESC256, 1u);
                            if (has_lo) tc_mma(tacc, a_lo, b_hi, IDESC256, 1u);
                        }
                        tc_commit(bar_empty + 8 * s);
                    }
                    tc_commit(bar_accf + 8 * buf);
                }
            }
        }
    } else {
        const int q = warp & 3;
        const int grp = (warp - 2) >> 2;
        const int r128 = q * 32 + lane;
        const int row = mt * BM + r128;
        const bool valid = row < G.M;
        const float *bias = G.bias[dir];
        uint32_t it = 0;
        for (int t = 0; t < G.T; t++) {
            const int tt = dir ? G.T - 1 - t : t, tp = dir ? tt + 1 : tt - 1;
            for (int nt = 0; nt < 2; nt++, it++) {
                const uint32_t buf = it & 1u, use = it >> 1;
                const int ubase = nt * (PBN / 4) + grp * (PG_COLS / 4);
                // previous hidden values of this thread's units (own writes of step t-1, or h0)
                float hp[PG_COLS / 4];
#pragma unroll
                for (int u8 = 0; u8 < PG_COLS / 32; u8++) {
                    uint4 h = make_uint4(0, 0, 0, 0), l = make_uint4(0, 0, 0, 0);
                    if (valid) {
                        const int j0 = ubase + u8 * 8;
                        const int64_t rel = (int64_t) (j0 >> 5) * TILE_ELEMS + ((j0 & 31) >> 3) * 1024 + r128 * 8;
                        const int64_t o = t == 0 ? (int64_t) mt * G.h0_mt_stride + rel : (int64_t) mt * seq_stride + ((int64_t) tp * 8 + dir * 4) * TILE_ELEMS + rel;
                        h = *reinterpret_cast<const uint4 *>((t == 0 ? G.h0_hi[dir] : G.y_hi) + o);
                        l = *reinterpret_cast<const uint4 *>((t == 0 ? G.h0_lo[dir] : G.y_lo) + o);
                    }
                    const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
                    for (int e = 0; e < 8; e++)
                        hp[u8 * 8 + e] = op_val(hw[e >> 1] >> (16 * (e & 1))) + op_val(lw[e >> 1] >> (16 * (e & 1)));
                }
                mbar_wait(bar_accf + 8 * buf, use & 1u);
                tc_fence_after();
#pragma unroll
                for (int cl = 0; cl < PG_COLS / 32; cl++) {
                    const int cc = grp * (PG_COLS / 32) + cl;
                    const int col0 = nt * PBN + cc * 32;
                    uint32_t acc[32];
                    tmem_ld32(tmem_base + buf * PBN + ((uint32_t) (q * 32) << 16) + (uint32_t) (cc * 32), acc);
                    if (cl == PG_COLS / 32 - 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(bar_acce + 8 * buf);
                    }
                    const int j0 = col0 >> 2;
                    float hn[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        const float4 bz = __ldg(reinterpret_cast<const float4 *>(bias + col0 + 4 * u));
                        const float v0 = __uint_as_float(acc[4 * u + 0]) + bz.x, v1 = __uint_as_float(acc[4 * u + 1]) + bz.y;
                        const float v2 = __uint_as_float(acc[4 * u + 2]) + bz.z, v3 = __uint_as_float(acc[4 * u + 3]) + bz.w;
                        const float r = sigm(v0), z = sigm(v1);
                        const float n = tanh_fast(v2 + r * v3);
                        hn[u] = (1.0f - z) * n + z * hp[cl * 8 + u];
                    }
                    if (valid) {
                        uint4 hi, lo;
                        split8(hn, hi, lo);
                        const int64_t o = (int64_t) mt * seq_stride + ((int64_t) tt * 8 + dir * 4 + (j0 >> 5)) * TILE_ELEMS + ((j0 & 31) >> 3) * 1024 + r128 * 8;
                        *reinterpret_cast<uint4 *>(G.y_hi + o) = hi;
                        *reinterpret_cast<uint4 *>(G.y_lo + o) = lo;
                    }
                }
                if (nt == 1) {
                    __threadfence();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_h);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t) PTMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------- operand preparation kernels
// int8 images [B][T][F] -> tiled operand [mt][T][1 k-tile] (hi only; |v| <= 128 is exact in bf16), and when op8 is set its
// e4m3 image (the a_hi operand of the a_hi*w_lo correction; e4m3 rounds |v| > 16 to 4 significant bits, ~2^-16 of the product)
__global__ void k_tc_pack_images(const int8_t *__restrict__ img, op_t *__restrict__ op, uint8_t *__restrict__ op8, int64_t B, int T, int F) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;     // one thread per (row, t, kc)
    const int64_t total = ceil_div(B, 128) * 128 * T * 4;
    if (i >= total) return;
    const int kc = (int) (i & 3);
    const int64_t rt = i >> 2;
    const int t = (int) (rt % T);
    const int64_t row = rt / T;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; e++) {
        const int k = kc * 8 + e;
        v[e] = (row < B && k < F) ? (float) img[(row * T + t) * F + k] : 0.f;
    }
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; i++) w[i] = (uint32_t) op_bits(v[2 * i]) | ((uint32_t) op_bits(v[2 * i + 1]) << 16);
    const int64_t tile = ((row >> 7) * T + t) * TILE_ELEMS;
    *reinterpret_cast<uint4 *>(op + tile + kc * 1024 + (row & 127) * 8) = make_uint4(w[0], w[1], w[2], w[3]);
    if (op8)
        *reinterpret_cast<uint2 *>(op8 + tile + (kc >> 1) * 2048 + (row & 127) * 16 + (kc & 1) * 8) =
            make_uint2(f8x2(v[0], v[1]) | (f8x2(v[2], v[3]) << 16), f8x2(v[4], v[5]) | (f8x2(v[6], v[7]) << 16));
}

}  // namespace tc
}  // namespace pb
