// Opaque handle layouts shared by the translation units of libpepper_b200.
#pragma once
#include "common.cuh"
#include <vector>

namespace pb {
struct VariantStream;      // streaming session state (pipeline.cu)
struct DevRnn { DevBuf W, bias; int K0, K0p, K1, Kp, H; };
struct DevLin { DevBuf W, bias; int N, K, Kp; };
// tcgen05 path (nets_tc.cu): weights as bf16 hi/lo tile images + per-chunk tiled operands
// with_f8 uploads (variant) also hold e4m3 images, and their fp16 images are scaled: accumulator x acc_scale = GEMM value
// (tc_gemm.cuh, "e4m3 correction operands")
struct TcRnn { DevBuf w_hi, w_lo, w8_hi, w8_lo; float acc_scale = 1.f; int nkt_x = 0, nkt_h = 0; };
struct TcLin { DevBuf w_hi, w_lo, w8_hi, w8_lo; float acc_scale = 1.f; int nkt = 0; };
struct TcVariant {
    TcRnn enc[2], dec[2];
    TcLin lin[5];
    DevBuf img_op, yenc_hi, yenc_lo, ydec_hi, ydec_lo, c, act_hi[2], act_lo[2], final_f32;
    DevBuf img_op8, yenc_hi8, yenc_lo8, ydec_hi8, ydec_lo8, act_hi8[2], act_lo8[2];      // e4m3 images of the same operands
    // which GEMMs execute the third (a_lo x w_hi) product: bit 0 encoder h-part, 1 decoder x-part, 2 decoder h-part, 3 linear_1,
    // 4 linear_2..5; clearing a bit runs that GEMM with two products, 0x1f = three everywhere.  Default 0x1a: the recurrent
    // (h-part) GEMMs of both LSTM layers run with two products — each passes the parity gate on its own (hidden states within
    // 1e-3, class index exact outside the 1e-4 margin; DESIGN.md section 4 has the per-GEMM errors) — while the decoder's x-part
    // and the MLP head, which fail it, keep three.
    int lo_mask = 0x1a;
    // same bit order: a set bit runs that GEMM's correction products (a_hi x w_lo, and a_lo x w_hi where lo_mask keeps it) as
    // e4m3 MMAs instead of fp16 ones.  0 = the fp16 split everywhere (the cross-check).
    int f8_mask = 0x1f;
};
struct TcPolish {
    TcRnn enc[2], dec[2];
    DevBuf img_op, yenc_hi, yenc_lo, ydec_hi, ydec_lo, zero, flags;
    int lo_mask = 0x7;      // bit 0 encoder h-part, 1 decoder x-part, 2 decoder h-part
};
// optional record sink of the variant head kernel: the encoder's columns of the candidates of this forward call + output records
struct OutSink {
    pb_candidate_columns_t cols{nullptr, nullptr, nullptr, nullptr, nullptr};
    pb_pred_record_t *records = nullptr;
    OutSink at(int64_t b0) const {
        OutSink S = *this;
        if (records) {
            S.cols.positions += b0; S.cols.region_of += b0; S.cols.depths += b0; S.cols.freqs += b0; S.cols.keys += b0 * PB_ALLELE_STRIDE;
            S.records += b0;
        }
        return S;
    }
};
int tc_upload_rnn(TcRnn &T, const float *Wp, int K0, int K0p_src, int H, int Kp_src, bool with_f8);
int tc_upload_lin(TcLin &T, const float *w, int N, int K, bool with_f8);
}  // namespace pb

struct pb_variant_encoder {
    int device = 0;
    pb::DevBuf op_ref, op_rd, read_reflen, read_region, tile_region, tile_x0, region_goff, M16, cov, meta, dbg,
        tile_nsites, tile_nev, tile_site_base, tile_ev_base, site_of, site_g, site_evoff, site_cur, ev, cand_tmp,
        site_ncand, site_region, site_candoff, rare, scalars;
    // host-entry staging
    pb::DevBuf h_pos, h_seq_off, h_cigar_off, h_flags, h_mapq, h_seq, h_qual, h_cigar, h_regions, h_ref;
    pb::DevBuf o_images, o_positions, o_depths, o_freqs, o_keys, o_region_of, o_per_region;
    cudaEvent_t evt[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    float ms[5] = {0, 0, 0, 0, 0};
    bool debug = false;
    // last-call bookkeeping for the debug read-back
    std::vector<int64_t> last_goff;
    std::vector<pb_region_t> last_regions;
    const char *last_d_ref = nullptr;
    size_t rare_cap = 1 << 20;
    // fused call scratch (pipeline.cu)
    pb::DevBuf p_images, p_positions, p_depths, p_freqs, p_keys, p_region_of, p_probs, p_per_region;
    cudaEvent_t pevt[3] = {nullptr, nullptr, nullptr};
    float pms[2] = {0, 0};
    int64_t launches = 0;
    // pipelined host entry (pipeline.cu): double-buffered staging + copy stream
    pb::DevBuf g_buf[2][10];
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t copied[2] = {nullptr, nullptr};
    pb::VariantStream *vstream = nullptr;
};

struct pb_polish_encoder {
    int device = 0;
    pb::DevBuf op_ref, op_rd, read_reflen, read_region, tile_region, tile_x0, region_goff, basecnt, cov, longest, tile_ncols,
        tile_col_base, col_of, inscnt, scalars;
    pb::DevBuf h_pos, h_seq_off, h_cigar_off, h_flags, h_mapq, h_seq, h_qual, h_cigar, h_regions;
    pb::DevBuf o_image, o_pos, o_idx, o_col_off;
    cudaEvent_t evt[4] = {nullptr, nullptr, nullptr, nullptr};
    float ms[3] = {0, 0, 0};
    // fused call scratch (pipeline.cu)
    pb::DevBuf p_image, p_pos, p_idx, p_col_off, p_chunks, p_imgs, p_position, p_index, p_bases, p_phred, p_iregion, p_cid;
    cudaEvent_t pevt[3] = {nullptr, nullptr, nullptr};
    float pms[2] = {0, 0};
    int64_t launches = 0;
};

struct pb_variant_net {
    int device = 0;
    int mode = 1;          // 1 = tcgen05 bf16x3 (default), 0 = fp32 FFMA
    pb::TcVariant *tc = nullptr;
    pb::DevRnn enc[2], dec[2];
    pb::DevLin lin[5], outl;
    // scratch for one chunk
    int64_t chunk = 0;
    pb::DevBuf h[2], c, yenc, ydec, l[2], img, probs;
    int64_t launches = 0;
};

struct pb_polish_net {
    int device = 0;
    int mode = 1;          // 1 = tcgen05 bf16x3 (default), 0 = fp32 FFMA
    pb::TcPolish *tc = nullptr;
    pb::DevRnn enc[2], dec[2];
    pb::DevBuf dW, dB;
    int64_t chunk = 0;
    pb::DevBuf h[2], yenc, ydec, acc, img, bases, phred;
    int64_t launches = 0;
};

namespace pb {
int variant_forward_tc(pb_variant_net *N, const int8_t *d_images, int64_t B, float *d_probs, float *d_hidden_dbg, cudaStream_t st,
                       void (*out_kernel)(const float *, const float *, const float *, float *, int64_t, const OutSink &, cudaStream_t),
                       const OutSink &sink);
int polish_forward_tc(pb_polish_net *N, const uint8_t *d_images, int64_t B, int64_t n_total, int64_t b0, float *d_hidden_dbg,
                      cudaStream_t st);
}  // namespace pb
