// Internal launcher interface shared by the translation units of libb200vad.so.
#pragma once
#include "common.cuh"
#include "../../include/b200vad.h"

namespace b200vad {

struct GemmArgs {
    const void* A;
    int64_t lda, rows_per_batch, a_batch_stride;   // in elements of A
    int64_t M;
    int N, K, Kp;                                   // Kp = K rounded up to 32 (W row stride)
    const __half* W_hi;
    const __half* W_lo;
    const float* bias;
    void* C;
    int64_t ldc;
    int c_half;                                     // 1: write fp16, 0: fp32
    int act;                                        // 0 none, 1 leaky_relu(0.01), 2 abs
};

int gemm_launch(const GemmArgs& a, int a_half, int terms, cudaStream_t stream);
// gate_scale != 0: rows are LSTM gate rows (i,f,g,o blocks of 128) and are pre-multiplied by lstm_gate_scale(row)
int split_weights(const float* w, int N, int K, int Kp, __half* hi, __half* lo, cudaStream_t stream, int gate_scale = 0);
int fbank_tables_init(int device);
int zero_f64_launch(double* p, int64_t n, cudaStream_t stream);
// rows != nullptr: row b starts at rows[b] (B device pointers of the sample type) instead of wav + b * stride
int fbank_launch(const void* wav, int wav_i16, const int32_t* lens, int B, int64_t N, int64_t stride, float* feats, __half* feats_hi,
                 __half* feats_lo, int64_t T_out, double* row_sums, int device, cudaStream_t stream, const void* const* rows = nullptr);
int lstm_recurrent_launch(const float* xg, const __half* whh, float* y, int B, int T, cudaStream_t stream);
int lstm_tc_set_tile(int nb);
// Scale s of the (x1, x2) activation planes of the 2-MMA projection: x1 = fp16((1 - s) x), x2 = fp16(x - x1) (gemm_tc.cu)
constexpr float kPlaneScale = 0.015625f;   // 2^-6
int lstm_tc_launch(const float* xg, const __half* whh, __half* y_hi, __half* y_lo, int B, int T, int scaled_planes, cudaStream_t st);
int gemm_ts_launch(const __half* a_hi, const __half* a_lo, int64_t lda, int64_t M, int K, const __half* w_hi, const __half* w_lo,
                   int Kp, int ldw, int N, const float* bias, int mode, int accumulate, float* c, __half* o_hi, __half* o_lo,
                   int64_t ldc, int num_sms, cudaStream_t st, const float* wc = nullptr, const float* bc = nullptr);
int gemm_ts_rows_launch(const __half* a_hi, const __half* a_lo, int64_t row_stride, int64_t batch_stride, int B, int rows_per_batch,
                        int K, const __half* w_hi, const __half* w_lo, int Kp, int ldw, int n_valid, const float* bias,
                        int accumulate, int act_abs, float* c, int64_t ldc, int64_t out_batch_rows, int out_row_step,
                        int out_row_off, int num_sms, cudaStream_t st);
int gemm_xg2_launch(const __half* x_hi, const __half* x_lo, int64_t lda, int B, int T, int K, const __half* w_hi,
                    const __half* w_lo, int Kp, int ldw, const float* bias, int terms, float* xg, int* sync,
                    size_t sync_bytes, int num_sms, cudaStream_t st);
int sinc_pool_gemm_launch(const __half* wn_hi, const __half* wn_lo, int64_t Np, int B, int64_t L1, const __half* w_hi,
                          const __half* w_lo, int Kp, int ldw, int n_valid, int terms, float* pooled, int ldc, double* stats,
                          int num_sms, cudaStream_t st);
int conv_pool_gemm_launch(const __half* a_hi, const __half* a_lo, int64_t row_stride, int64_t batch_stride, int B, int64_t L, int K,
                          const __half* w_hi, const __half* w_lo, int Kp, int ldw, int n_valid, const float* bias, int terms,
                          float* pooled, int ldc, double* stats, int num_sms, cudaStream_t st);
int head_fused_launch(const __half* y_hi, const __half* y_lo, int64_t M, const __half* w1_hi, const __half* w1_lo, const __half* w2_hi,
                      const __half* w2_lo, const float* b1, const float* b2, const float* wc, const float* bc, float* prob, int num_sms,
                      cudaStream_t st);
int gemm_xg_pair_launch(const __half* x_a, const __half* x_b, int64_t lda, int B, int T, int K, const __half* w_hi,
                        const __half* w_lo, int Kp, int ldw, const float* bias, int terms, float* xg, int* sync,
                        size_t sync_bytes, int num_sms, cudaStream_t st);
int gemm_ts_xg_launch(const __half* x_hi, const __half* x_lo, int64_t lda, int B, int T, int K, const __half* w_hi,
                      const __half* w_lo, int Kp, int ldw, const float* bias, int accumulate, float* xg, int num_sms,
                      cudaStream_t st);
int split_planes_pad_launch(const float* x, int64_t rows, int D, int D8, __half* hi, __half* lo, cudaStream_t st);
int split_planes_launch(const float* x, int64_t n, __half* hi, __half* lo, cudaStream_t st);
int classifier_launch(const float* z, int64_t rows, const float* wc, const float* bc, float* prob, cudaStream_t stream);
int pack_whh(const float* w, __half* out, cudaStream_t stream, __half* out_lo = nullptr);
// fused projection + recurrence on 4-CTA clusters (lstm_fused.cu); D <= 256
int lstm_fused_supported(int D);
int lstm_fused_clusters();
void lstm_fused_set_debug(int flags, int lag);
int lstm_fused_read_debug(long long* host, int n);
int lstm_fused_last_timeout(int* out7);
int lstm_fused_launch(const __half* x_a, const __half* x_b, int64_t lda, int B, int T, int D, const __half* wih_hi,
                      const __half* wih_lo, int ldw, const __half* whh_hi, const __half* whh_lo, const float* bias, int terms,
                      __half* y_a, __half* y_b, int y_scaled, cudaStream_t st);
// the same layer with every product issued as cta_group::2 MMAs by CTA pairs (lstm_pair.cu): half the operand traffic per CTA
int lstm_pair_launch(const __half* x_a, const __half* x_b, int64_t lda, int B, int T, int D, const __half* wih_hi,
                     const __half* wih_lo, int ldw, const __half* whh_hi, const __half* whh_lo, const float* bias, int terms,
                     __half* y_a, __half* y_b, cudaStream_t st);
int lstm_pair_last_timeout(int* out7);
void lstm_pair_set_opt(int opt);
int lstm_pair_read_debug(long long* host, int n);
int add_bias(const float* a, const float* b, float* out, int n, cudaStream_t stream);
// stream_off == nullptr: B rows of T frames; else B streams prob[stream_off[b], stream_off[b + 1]) of at most T frames each, written
// at the same offsets of out
int threshold_median_launch(const float* prob, int B, int64_t T, float thr, int kernel, void* out, int elem,
                            int32_t* near_count, float near_tol, cudaStream_t stream, const int64_t* stream_off = nullptr);
// offsets == nullptr: R uniform rows of uniform_T frames
int segments_launch(const uint8_t* dec, const int64_t* offsets, int64_t uniform_T, int R, int min_run, int row_base,
                    int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap, cudaStream_t stream);
// offsets == nullptr: R rows of T frames; else T = frames of the flat buffer (dec is written over [0, T)).  p is validated.
int binarize_launch(const float* prob, const int64_t* offsets, int64_t T, int R, const b200vad_binarize_params& p, int row_base,
                    uint8_t* dec, int32_t* counts, int64_t* seg_off, int32_t* seg, int64_t cap, cudaStream_t stream);
// b200vad_regions_step on validated arguments (prob may be null when nf == 0)
int regions_step_launch(const float* prob, int S, int nf, int64_t row_stride, const b200vad_binarize_params& p, int64_t* state,
                        const uint8_t* flush, int64_t* ev, int32_t* ev_counts, int64_t cap, cudaStream_t stream);
int sinc_filters_launch(const float* low, const float* band, const float* window, const float* n, float* out, cudaStream_t s);
int repack_conv_launch(const float* w, int Cout, int Cin, int k, float* out, cudaStream_t s);
int wave_instnorm_launch(const float* wav, int B, int64_t N, int64_t stride, const float* gamma, const float* beta,
                         double* stats, float* out, cudaStream_t s);
int norm_lrelu_launch(float* pooled, int B, int64_t P, int C, const double* stats, const float* gamma, const float* beta,
                      cudaStream_t s, __half* p_hi = nullptr, __half* p_lo = nullptr, int Cp = 0, int scaled_planes = 0);
int pool_norm_lrelu_launch(const float* in, int B, int64_t L, int C, float* pooled, double* stats, const float* gamma,
                           const float* beta, cudaStream_t s, __half* p_hi = nullptr, __half* p_lo = nullptr, int Cp = 0, int scaled_planes = 0);
// wav: (B, N) f32 rows, or int16 PCM rows (wav_i16 != 0; samples int16 / 32768), `stride` elements apart.  rows != nullptr: row
// b starts at rows[b] instead, and lens[b] (required with rows) are its valid samples; samples at index >= lens[b] read as 0
int wave_norm_planes_launch(const void* wav, int wav_i16, int B, int64_t N, int64_t stride, int64_t Np, const float* gamma,
                            const float* beta, double* stats, __half* hi, __half* lo, cudaStream_t s, int scaled_planes = 0,
                            const void* const* rows = nullptr, const int32_t* lens = nullptr);
int pad_rows_launch(const float* w, int Cout, int K, int ld, float* out, cudaStream_t s);
int repack_conv_pad_launch(const float* w, int Cout, int Cin, int k, int Cp, int ld, float* out, cudaStream_t s);

int stat_scores_launch(const uint8_t* dec, const uint8_t* lab, int64_t n, int64_t* out4, cudaStream_t st);
int score_intervals_launch(const int32_t* gt_iv, int64_t n_gt, const int32_t* pred_iv, int64_t n_pred, const int64_t* word_off,
                           const int32_t* nframes, int R, int64_t total_words, uint32_t* masks, int64_t* fa, int64_t* md,
                           int max_words_per_rec_hint, cudaStream_t st);
// win_off == nullptr: one recording of W windows and L frames; else R recordings, windows [win_off[r], win_off[r + 1]) of prob
// stitched into out[frame_off[r], frame_off[r + 1]), each at most L frames.  elem: 4 (f32) or 1 (u8)
int stitch_center_launch(const void* prob, const int64_t* win_off, const int64_t* frame_off, int R, int W, int Tw, int hop, void* out,
                         int64_t L, int elem, cudaStream_t st);
int stream_append_launch(float* ring, const float* chunk, float* lin, int S, int Wn, int hop, int pos, cudaStream_t st);
int stream_newest_launch(const float* prob, const uint8_t* dec, int S, int64_t T, int nf, float* prob_out, uint8_t* dec_out,
                         cudaStream_t st);
int synth_corpus_launch(float* out, int64_t utt0, int rows, int64_t N, uint64_t seed, cudaStream_t st);

}  // namespace b200vad
