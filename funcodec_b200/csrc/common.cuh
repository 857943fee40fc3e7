// Shared device/host definitions for the funcodec_b200 kernels (sm_100a).
//
// HBM layout (DESIGN.md section 3): every activation is stored CHANNELS-LAST, [B][T][C] fp32, RAW
// (= conv output incl. bias, before GroupNorm).  GroupNorm(1,C) needs the statistics of the whole
// (C x T) plane of a clip, so a layer cannot normalise its own output in its epilogue; instead each
// conv emits per-CTA (sum, sum^2) partials, a tiny finalize kernel turns them into (mean, rstd) per
// clip, and the CONSUMER applies   y = x * (rstd*gamma[c]) + (beta[c] - mean*rstd*gamma[c])
// (ATen's GroupNorm formulation) + optional second operand (resblock sum) + optional ELU while it
// stages its input tile into shared memory.  No normalised tensor is ever written to HBM.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace fcb {

// A (possibly normalised) view of a raw activation tensor.
struct InView {
    const float* x;          // raw [B][rows][C]; nullptr => view unused
    const float* stats;      // [B][2] = (mean, rstd); nullptr => identity (plain tensor)
    const float* gamma;      // [C] GroupNorm weight (used when stats != nullptr)
    const float* beta;       // [C] GroupNorm bias
    const float* coef;       // [B][2][C] precomputed (rstd*gamma, beta - mean*rstd*gamma) or nullptr (identity)
    long long clip_stride;   // elements between consecutive clips
    int row_off;             // first logical row (transposed-conv trim, conv.py:299-303)
};

// conv_tc.cu, FreqCodec 2-D mode (KF > 0): every (clip, output frequency row) is a pseudo-clip of a conv along time
// whose input channels are the KF frequency taps x cin channels, gathered from KF input rows [B][F_raw][T_raw][cin].
struct Freq2d {
    int KF, SF, pad_f;       // frequency taps, stride, leading padding (KF == 0: plain 1-D conv)
    int F_in, F_out;         // logical input rows, output rows (= pseudo-clips per clip)
    int cin;                 // channels of the stored input (ConvParams::C_in is the gathered KF*cin)
    int T_raw0, T_raw1;      // allocated time extents of in0 / in1 (InView::row_off = first logical column)
    int f_off0, f_off1;      // first logical frequency row of in0 / in1
    int FR, TR, Cc;          // transposed conv phase scatter: output channel co -> phase co / Cc = pf*TR + pt
    int c_store;             // channels per stored output element (== Cc unless the weight image pads C_out)
};

struct ConvParams {
    InView in0, in1;         // input = f(in0) [+ f(in1)]   (resblock: shortcut + block)
    const float* div_scale;  // [B] or nullptr: input = x / scale[b]  (codec_basic.py:366-371)
    int elu;                 // apply ELU(alpha=1) to the summed input
    int T_in, C_in;
    int K, S, D;             // taps, stride, dilation
    int pad_l;               // left padding
    int T_ext;               // reflect period length (== T_in unless the tiny-input branch, conv.py:89-97)
    int pad_zero;            // 1: out-of-range taps read 0 (transposed conv as 2-tap conv); 0: reflect
    const float* w;          // packed [K][C_in][C_out]
    const float* w_tc;       // tensor-core image (conv_tc.cu) or nullptr
    int n_tile;              // output channels per CTA on the tensor-core path
    float tc_w_scale;        // power-of-two scale baked into the w_tc image (engine.cu build_tc_image_f16)
    float tc_in_scale;       // tensor-core path: power-of-two scale of the fp16-split activation operand (0 -> default 16)
    float tc_out_scale;      // 1 / (tc_in_scale * weight scale of the layer's image): applied to the accumulator in the epilogue
    float tc_elu_k;          // log2(e) / tc_in_scale (set by launch_conv_tc)
    const float* bias;       // [C_out]
    float* out;              // raw [B][T_out][C_out]
    int T_out, C_out;
    long long out_clip_stride;
    double* partials;        // [B][n_parts][2] (sum, sum of squares) or nullptr
    int cic;                 // input-channel chunk staged per iteration
    Freq2d fq;               // tensor-core 2-D mode (zero-initialised for 1-D layers)
};

// ---- FreqCodec 2-D path (conv2d_simt.cu): raw activations are channels-last [B][F_raw][T_raw][C]
struct InView2 {
    const float* x;          // nullptr => view unused
    const float* coef;       // [B][2][C] deferred-GroupNorm affine or nullptr (plain tensor)
    int F_raw, T_raw;        // allocated extents
    int f_off, t_off;        // first logical frequency row / time column (transposed-conv trim, conv.py:430-445)
};

struct Conv2dParams {
    InView2 in0, in1;
    int elu;
    int B, F_in, T_in, C_in; // logical input extents
    int KF, KT, SF, ST;      // taps and strides per axis (dilation 1)
    int pad_f, pad_t;        // leading padding per axis (time: incl. the extra padding, conv.py:368)
    int pad_zero;            // 1: transposed conv as 2x2-tap zero-padded conv; 0: reflect
    const float* w;          // packed [KT][KF*C_in][C_out_eff]
    const float* bias;       // [C_out_eff]
    float* out;              // raw [B][F_out*FR][T_out*TR][Cc]
    int F_out, T_out, C_out_eff;
    int FR, TR, Cc;          // phase scatter of a transposed conv (C_out_eff = FR*TR*Cc); plain conv: 1, 1, C_out
    double* partials;        // [B*F_out][n_parts][2] or nullptr
    int cic;
};

__device__ __forceinline__ float elu1(float v) {
    // ATen CPU ELU: x <= 0 ? (exp(x) - 1) : x   (alpha = 1)
    return v > 0.f ? v : (expf(v) - 1.0f);
}

__device__ __forceinline__ int reflect_index(int i, int n) {
    // F.pad(mode='reflect') index map for one reflection (|pad| < n is guaranteed by the caller)
    if (i < 0) i = -i;
    if (i >= n) i = 2 * (n - 1) - i;
    return i;
}

// Block-wide sum of two doubles (deterministic order).  red must hold 2*32 doubles.
__device__ __forceinline__ void block_reduce_2d(double& a, double& b, double* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (lane == 0) { red[warp] = a; red[32 + warp] = b; }
    __syncthreads();
    if (warp == 0) {
        a = lane < nwarps ? red[lane] : 0.0;
        b = lane < nwarps ? red[32 + lane] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
        }
    }
}

}  // namespace fcb
