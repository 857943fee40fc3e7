// Host-callable launchers of the funcodec_b200 kernels (all asynchronous on the given stream).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

namespace fcb {

// misc.cu: opt a kernel in to `bytes` of dynamic shared memory once per (kernel, device); thread-safe.
cudaError_t ensure_dynamic_smem(const void* kernel, int bytes);

// conv_simt.cu
void conv_pick_tile(int T_out, int C_out, int C_in, int K, int B, int* tx, int* tm, bool* two);
int conv_num_parts(int T_out, int C_out, int C_in, int K, int B);
cudaError_t launch_conv(const ConvParams& p, int B, cudaStream_t st, int* nparts);
cudaError_t launch_stats_finalize(const double* partials, int nparts, double count, float eps, int mode,
                                  float* out, int B, cudaStream_t st, const float* gamma = nullptr,
                                  const float* beta = nullptr, int C = 0, float* coef = nullptr);
bool conv_cout1_supported(const ConvParams& p);          // C_out 1 or 2 (mono / stereo decoder output conv)
int conv_cout1_num_parts(int T_out, int C_out);
cudaError_t launch_conv_cout1(const ConvParams& p, int B, cudaStream_t st, int* nparts);
int sumsq_num_parts(int L);
// C = 2: planar stereo clips [B][2][L], squares of the mono mix (x0 + x1) / 2
cudaError_t launch_sumsq_partials(const float* x, int B, int L, double* partials, int* nparts, cudaStream_t st, int C = 1);

// conv_tc.cu
bool conv_tc_supported(int C_in, int C_out_eff, int K, int S, int D);
bool conv_tc_supported_2d(int cin, int C_out_eff, int KT, int ST);
int conv_tc_n_tile(int C_out_eff);
int conv_tc_num_parts(int T_out, int C_out_eff);
cudaError_t launch_conv_tc(const ConvParams& p, int B, cudaStream_t st, int* nparts);

// conv2d_simt.cu (FreqCodec 2-D path)
int conv2d_num_parts(const Conv2dParams& p);
cudaError_t launch_conv2d(const Conv2dParams& p, cudaStream_t st);
bool conv2d_small_cout_supported(const Conv2dParams& p);          // C_out <= 4 stride-1 conv (halo tile, FMA-bound)
int conv2d_small_cout_num_parts(const Conv2dParams& p);
cudaError_t launch_conv2d_small_cout(const Conv2dParams& p, cudaStream_t st);
cudaError_t launch_stft_magphase(const float* wav, const float* scale, int B, int L, int n_fft, int hop, int n_frames,
                                 int cpad, float* feats, cudaStream_t st);
cudaError_t launch_istft(const float* raw, const float* coef, int B, int F_raw, int T_raw, int n_fft, int hop, int n_frames,
                         const float* scale, float* frames, float* out, int out_len, cudaStream_t st);

// STFT / iSTFT as tensor-core GEMMs ("stft_tc" option, default on): the glue kernels around two conv_tc launches
cudaError_t launch_wave_rows(const float* wav, const float* scale, int B, int L, int n_fft, int n_rows, float* rows, cudaStream_t st);
cudaError_t launch_magphase_from_spec(const float* spec, int ld, int B, int n_bins, int n_frames, int cpad, float* feats,
                                      cudaStream_t st);
cudaError_t launch_spec_rows(const float* raw, const float* coef, int B, int F_raw, int T_raw, int n_bins, int n_frames, int ld,
                             float* Y, cudaStream_t st);
cudaError_t launch_istft_ola(const float* frames, const float* scale, int B, int n_fft, int hop, int n_frames, int out_len,
                             float* out, cudaStream_t st);

// lstm.cu
struct LstmSeqParams {
    const float* gx;      // [B][T][4H] input projection incl. both biases, columns packed unit-major (n' = 4*j + gate)
    const float* whh;     // [H][4H] packed W_hh^T, same column order
    float* h_seq;         // [B][T][H] hidden states of this layer
    float* y_out;         // nullptr, or [B][T][H]: y = h + skip   (SLSTM skip, lstm.py:25-26)
    InView skip;          // the SLSTM input (normalised on load) when y_out != nullptr
    unsigned* barrier;    // device counter for the per-step grid barrier (zeroed by the launcher)
    int B, T, H;
    float whh_scale, whh_inv_scale;   // tensor-core gate GEMM: power-of-two operand scale of W_hh and 1 / (whh_scale * 4096) (0: fp32 path)
    unsigned long long* trace;   // PROFILING ONLY (env FCB_LSTM_TRACE): [LSTM_TRACE_ITEMS][8] %globaltimer stamps of CTA 0, or nullptr
};
constexpr int LSTM_TRACE_ITEMS = 64, LSTM_TRACE_FIRST_STEP = 100;
cudaError_t launch_lstm_seq(const LstmSeqParams& p, cudaStream_t st);
int lstm_pick_units(int H);

// rvq.cu
struct RvqParams {
    InView in;            // encoder output view [B][T'][D] (normalised on load)
    const float* embed;   // [n_q_max][K][D]
    const float* cnorm;   // [n_q_max][K]  |c|^2
    const float* embed_tc; // tensor-core image of the codebooks (rvq_tc.cu) or nullptr
    int B, T, D, K, n_q;
    long long* codes;     // [n_q][B][T]
    float* quant;         // [B][T][D] or nullptr
    float* sub_quants;    // [n_q][B][D][T] or nullptr
    float* enc_out;       // [B][T][D] or nullptr
    int allow_sliced;     // rvq_simt.cu: permit the column-sliced kernel for a D too wide for the whole-chunk one ("rvq_sliced" option)
};
cudaError_t launch_rvq(const RvqParams& p, cudaStream_t st);
int rvq_simt_slice(int D);      // 0: no SIMT RVQ kernel for this D; D: whole-chunk kernel; else the sliced kernel's slice width
constexpr int RVQ_TC_N = 128;   // codewords per tensor-core tile == n_tile of the codebook slab image
bool rvq_tc_supported(int D, int K);
cudaError_t launch_rvq_tc(const RvqParams& p, cudaStream_t st);
cudaError_t launch_code_norms(const float* embed, float* cnorm, int rows, int D, cudaStream_t st);
cudaError_t launch_embed_sum(const long long* codes, int q_major, const float* embed, int B, int T, int n_q, int K, int D,
                             float* out, int* err_flag, cudaStream_t st);

// misc.cu
// raw [B][T_raw][C] channels-last -> out [B][C][out_len] planar, C in {1, 2}
cudaError_t launch_final_output(const float* raw, const float* stats, const float* gamma, const float* beta,
                                const float* scale, int B, int T_raw, int out_len, float* out, cudaStream_t st, int C = 1);
cudaError_t launch_fill(float* p, float v, long long n, cudaStream_t st);
// planar multi-channel clips [B][C][L] are B*C rows here (segments [(s*B + b)][C][seg_len]); launch_overlap_add likewise
cudaError_t launch_gather_segments(const float* wav, int B, int L, int seg_len, int stride, int s0, int n_seg, float* out,
                                   cudaStream_t st);
constexpr int OLA_MAX_TAILS = 16;
struct OlaParams {
    const float* full;                 // decoded full-length segments [(s*B + b)][dl0]
    const float* tail[OLA_MAX_TAILS];  // decoded shorter trailing segments [B][tail_dl[i]]
    int tail_dl[OLA_MAX_TAILS];
    int n_seg, n_full, dl0, stride, B, out_len;
    float* out;                        // [B][out_len]
};
cudaError_t launch_overlap_add(const OlaParams& p, cudaStream_t st);

}  // namespace fcb
