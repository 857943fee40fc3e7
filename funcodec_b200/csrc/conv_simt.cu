// Channels-last direct Conv1d (fp32 SIMT) with fused input transform and GroupNorm partial statistics.
//
// Replaces, for one layer, the reference sequence
//     [previous GroupNorm apply] -> [resblock add] -> [ELU] -> F.pad(reflect) -> Conv1d(bias) -> NaN check
//     (funcodec/modules/normed_modules/conv.py:243-261, :155-164; seanet_encoder.py:61)
// with ONE kernel: the input tile is normalised / summed / activated / reflect-indexed while it is
// staged into shared memory, the conv is a register-tiled (TM x 8) outer-product loop, and the epilogue
// adds the bias, stores the RAW output and emits this CTA's (sum, sum^2) for the layer's own GroupNorm.
// SConvTranspose1d (conv.py:281-305) runs through the same kernel as a 2-tap zero-padded conv with
// C_out' = stride * C_out (engine.cu packs the weights accordingly), and so do the LSTM input
// projections (1x1 conv == GEMM).
//
// Roofline: compute-bound on the fp32 FMA pipe for C_in*K >= ~128, HBM-bound for the C<=32 layers.
// Algorithmic bytes per launch = 4 * B * (T_in*C_in + T_out*C_out) (+ weights once).
#include "common.cuh"
#include "kernels.h"

namespace fcb {

template <int TX, int TM, bool TWO_LEVEL>
__global__ void __launch_bounds__(256, TWO_LEVEL ? 1 : 2) conv1d_cl_kernel(const ConvParams p) {
    constexpr int TN = 8;
    constexpr int TY = 256 / TX;
    constexpr int CO_TILE = TX * TN;
    constexpr int T_TILE = TY * TM;
    extern __shared__ __align__(16) float smem[];

    const int tid = threadIdx.x;
    const int tx = tid % TX, ty = tid / TX;
    const int b = blockIdx.z;
    const int t0 = blockIdx.x * T_TILE;
    const int co0 = blockIdx.y * CO_TILE;
    const int C_in = p.C_in, cic = p.cic, K = p.K, S = p.S, D = p.D;
    const int R = (T_TILE - 1) * S + (K - 1) * D + 1;
    const int pitch = cic + 1;
    const bool has1 = p.in1.x != nullptr;

    float* coefA0 = smem;
    float* coefB0 = coefA0 + C_in;
    float* coefA1 = coefB0 + C_in;
    float* coefB1 = coefA1 + (has1 ? C_in : 0);
    float* Ws = coefB1 + (has1 ? C_in : 0);
    Ws += (4 - ((Ws - smem) & 3)) & 3;                      // 16-byte align for float4 reads
    float* Xs = Ws + K * cic * CO_TILE;

    // ---- per-clip, per-channel GroupNorm coefficients (ATen: scale = rstd*gamma, bias = beta - scale*mean)
    {
        float mean0 = 0.f, rstd0 = 1.f, mean1 = 0.f, rstd1 = 1.f;
        if (p.in0.stats) { mean0 = p.in0.stats[2 * b]; rstd0 = p.in0.stats[2 * b + 1]; }
        if (has1 && p.in1.stats) { mean1 = p.in1.stats[2 * b]; rstd1 = p.in1.stats[2 * b + 1]; }
        for (int c = tid; c < C_in; c += 256) {
            float a = 1.f, bb = 0.f;
            if (p.in0.stats) { a = rstd0 * p.in0.gamma[c]; bb = p.in0.beta[c] - a * mean0; }
            coefA0[c] = a; coefB0[c] = bb;
            if (has1) {
                a = 1.f; bb = 0.f;
                if (p.in1.stats) { a = rstd1 * p.in1.gamma[c]; bb = p.in1.beta[c] - a * mean1; }
                coefA1[c] = a; coefB1[c] = bb;
            }
        }
    }
    const float inv_div = p.div_scale ? p.div_scale[b] : 1.f;   // used as a divisor (exact x / scale)
    const float* x0 = p.in0.x + (long long)b * p.in0.clip_stride + (long long)p.in0.row_off * C_in;
    const float* x1 = has1 ? p.in1.x + (long long)b * p.in1.clip_stride + (long long)p.in1.row_off * C_in : nullptr;
    const int gt_max = (p.T_out - 1) * S - p.pad_l + (K - 1) * D;   // last input position any valid output reads

    float acc[TM][TN];
    float tot[TWO_LEVEL ? TM : 1][TWO_LEVEL ? TN : 1];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
    if (TWO_LEVEL) {
#pragma unroll
        for (int i = 0; i < (TWO_LEVEL ? TM : 1); ++i)
#pragma unroll
            for (int j = 0; j < (TWO_LEVEL ? TN : 1); ++j) tot[i][j] = 0.f;
    }

    const int c_st = tid % cic;              // this thread's channel within the chunk (cic divides 256)
    const int r_st = tid / cic;
    const int r_step = 256 / cic;

    for (int ci0 = 0; ci0 < C_in; ci0 += cic) {
        __syncthreads();
        // ---- stage the transformed input window: Xs[row][c]
        {
            const int c = ci0 + c_st;
            const float a0 = coefA0[c], b0 = coefB0[c];
            const float a1 = has1 ? coefA1[c] : 0.f, b1 = has1 ? coefB1[c] : 0.f;
            for (int row = r_st; row < R; row += r_step) {
                const int gt = t0 * S - p.pad_l + row;
                float v = 0.f;
                bool ok = gt <= gt_max;
                int src = gt;
                if (p.pad_zero) ok = ok && gt >= 0 && gt < p.T_in;
                else { src = reflect_index(gt, p.T_ext); ok = ok && src < p.T_in; }
                if (ok) {
                    const long long off = p.in_ch_stride ? (long long)c * p.in_ch_stride + src : (long long)src * C_in + c;
                    float xv = __ldg(x0 + off);
                    if (p.div_scale) v = xv / inv_div;
                    else v = fmaf(xv, a0, b0);
                    if (has1) v = v + fmaf(__ldg(x1 + off), a1, b1);
                    if (p.elu) v = elu1(v);
                }
                Xs[row * pitch + c_st] = v;
            }
        }
        // ---- stage the weight chunk: Ws[k][c][co]
        for (int e = tid; e < K * cic * CO_TILE; e += 256) {
            const int j = e % CO_TILE;
            const int kc = e / CO_TILE;          // k * cic + c
            const int k = kc / cic, c = kc - k * cic;
            const int co = co0 + j;
            Ws[e] = co < p.C_out ? __ldg(p.w + ((long long)k * C_in + ci0 + c) * p.C_out + co) : 0.f;
        }
        __syncthreads();
        // ---- register-tiled FMA loop
        for (int c = 0; c < cic; ++c) {
            for (int k = 0; k < K; ++k) {
                const float* xr = Xs + (ty * S + k * D) * pitch + c;
                float a[TM];
#pragma unroll
                for (int i = 0; i < TM; ++i) a[i] = xr[i * TY * S * pitch];
                // a thread owns channels {4tx..4tx+3} and {CO_TILE/2 + 4tx..+3}: both float4 reads are contiguous
                // across the lanes of a warp (no bank conflicts), and so are the output stores
                const float* wrow = Ws + (k * cic + c) * CO_TILE + tx * 4;
                const float4 w0 = *reinterpret_cast<const float4*>(wrow);
                const float4 w1 = *reinterpret_cast<const float4*>(wrow + CO_TILE / 2);
#pragma unroll
                for (int i = 0; i < TM; ++i) {
                    acc[i][0] = fmaf(a[i], w0.x, acc[i][0]);
                    acc[i][1] = fmaf(a[i], w0.y, acc[i][1]);
                    acc[i][2] = fmaf(a[i], w0.z, acc[i][2]);
                    acc[i][3] = fmaf(a[i], w0.w, acc[i][3]);
                    acc[i][4] = fmaf(a[i], w1.x, acc[i][4]);
                    acc[i][5] = fmaf(a[i], w1.y, acc[i][5]);
                    acc[i][6] = fmaf(a[i], w1.z, acc[i][6]);
                    acc[i][7] = fmaf(a[i], w1.w, acc[i][7]);
                }
            }
        }
        if (TWO_LEVEL) {   // fold the chunk sum into the running total: short fp32 chains (DESIGN.md section 5)
#pragma unroll
            for (int i = 0; i < (TWO_LEVEL ? TM : 1); ++i)
#pragma unroll
                for (int j = 0; j < (TWO_LEVEL ? TN : 1); ++j) { tot[i][j] += acc[i][j]; acc[i][j] = 0.f; }
        }
    }

    // ---- epilogue: bias, raw store, GroupNorm partial statistics
    float s = 0.f, ss = 0.f;
    const int coA = co0 + tx * 4, coB = co0 + CO_TILE / 2 + tx * 4;    // channel of acc[.][0] and acc[.][4]
    float bias[TN];
#pragma unroll
    for (int j = 0; j < TN; ++j) {
        const int co = (j < 4 ? coA : coB - 4) + j;
        bias[j] = (co < p.C_out) ? __ldg(p.bias + co) : 0.f;
    }
    float* outb = p.out + (long long)b * p.out_clip_stride;
    const bool vec_ok = (p.C_out % 4 == 0);
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        const int t = t0 + ty + i * TY;
        if (t >= p.T_out) continue;
        float o[TN];
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int co = (j < 4 ? coA : coB - 4) + j;
            o[j] = (TWO_LEVEL ? tot[TWO_LEVEL ? i : 0][TWO_LEVEL ? j : 0] : acc[i][j]) + bias[j];
            if (co < p.C_out) { s += o[j]; ss = fmaf(o[j], o[j], ss); }
        }
        float* row = outb + (long long)t * p.C_out;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int co = half ? coB : coA;
            if (vec_ok && co + 4 <= p.C_out) {
                *reinterpret_cast<float4*>(row + co) = make_float4(o[4 * half], o[4 * half + 1], o[4 * half + 2], o[4 * half + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (co + j < p.C_out) row[co + j] = o[4 * half + j];
            }
        }
    }
    if (p.partials) {
        __shared__ double red[64];
        double ds = (double)s, dss = (double)ss;
        block_reduce_2d(ds, dss, red);
        if (tid == 0) {
            const int nparts = gridDim.x * gridDim.y;
            double* dst = p.partials + ((long long)b * nparts + blockIdx.y * gridDim.x + blockIdx.x) * 2;
            dst[0] = ds; dst[1] = dss;
        }
    }
}

// (mean, rstd) per clip from the per-CTA partials, fixed summation order (deterministic).
// GroupNorm(1, C): var is the biased variance over C*T elements; rstd = 1/sqrt(var + eps)
// (ATen group_norm CPU kernel).  mode 1: RMS scale of the input clip, 1e-8 + sqrt(mean(x^2))
// (funcodec/models/codec_basic.py:366-369).
__global__ void stats_finalize_kernel(const double* __restrict__ partials, int nparts, double count,
                                      float eps, int mode, float* __restrict__ out, const float* __restrict__ gamma,
                                      const float* __restrict__ beta, int C, float* __restrict__ coef) {
    __shared__ double red[64];
    const int b = blockIdx.x;
    double s = 0.0, ss = 0.0;
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) {
        s += partials[((long long)b * nparts + i) * 2];
        ss += partials[((long long)b * nparts + i) * 2 + 1];
    }
    block_reduce_2d(s, ss, red);
    __shared__ float mr[2];
    if (threadIdx.x == 0) {
        if (mode == 0) {
            const double mean = s / count;
            double var = ss / count - mean * mean;
            if (var < 0.0) var = 0.0;
            mr[0] = (float)mean;
            mr[1] = (float)(1.0 / sqrt(var + (double)eps));
            out[2 * b] = mr[0];
            out[2 * b + 1] = mr[1];
        } else {
            out[b] = 1e-8f + sqrtf((float)(ss / count));
        }
    }
    if (mode == 0 && coef) {      // per-channel affine of the deferred GroupNorm, consumed by the tensor-core producers
        __syncthreads();
        const float mean = mr[0], rstd = mr[1];
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            const float a = rstd * gamma[c];
            coef[(long long)b * 2 * C + c] = a;
            coef[(long long)b * 2 * C + C + c] = beta[c] - a * mean;
        }
    }
}

// Per-clip sum of squares partials of the raw waveform (for the RMS scale).  C = 2: the planar stereo clip [2][L]; the
// squares are those of the mono mix m = (x0 + x1) * 0.5 rounded to fp32 first, as x.mean(dim=1) is (codec_basic.py:366-368).
template <int C>
__global__ void sumsq_partials_kernel(const float* __restrict__ x, int L, int chunk, double* __restrict__ partials) {
    __shared__ double red[64];
    const int b = blockIdx.y;
    const int start = blockIdx.x * chunk;
    const int end = min(L, start + chunk);
    const float* xb = x + (long long)b * C * L;
    float s = 0.f, ss = 0.f;
    double ds = 0.0, dss = 0.0;
    int n = 0;
    for (int i = start + threadIdx.x; i < end; i += blockDim.x) {
        const float v = C == 1 ? xb[i] : __fmul_rn(__fadd_rn(xb[i], xb[(long long)(C - 1) * L + i]), 0.5f);
        s += v; ss = fmaf(v, v, ss);
        if (++n == 64) { ds += s; dss += ss; s = 0.f; ss = 0.f; n = 0; }
    }
    ds += s; dss += ss;
    block_reduce_2d(ds, dss, red);
    if (threadIdx.x == 0) {
        double* dst = partials + ((long long)b * gridDim.x + blockIdx.x) * 2;
        dst[0] = ds; dst[1] = dss;
    }
}

// Conv with one or two output channels (the decoder's last SConv1d, seanet_decoder.py:160-164; CO = 2 for a stereo decoder):
// pure HBM streaming (reads C_in floats per sample, writes CO).  out[t][co] = bias[co] + sum_k d_k,co[t + k - pad],
// d_k,co[r] = sum_c f(x[r][c]) w[k][c][co]: every input row is loaded (coalesced: 8 lanes x 16 B per row, 4 rows per warp
// instruction), transformed and dotted with the K x CO taps exactly ONCE -- each lane holds the K x 4 x CO weights of its 4
// channels in registers, the 8 lanes of a row reduce with 3 shuffle levels -- and the K x CO partial products per row go
// through shared memory to the threads that own the outputs.  The CTA's (sum, sum^2) covers all CO channels of its rows
// (GroupNorm(1, CO), conv.py:45-52).  C_in == 32, K <= 8; the time tile shrinks with CO to keep the static shared memory.
constexpr int C1_THREADS = 256, C1_TILE = 1024, C1_KMAX = 8;

template <int CO>
__global__ void __launch_bounds__(C1_THREADS) conv1d_cout1_kernel(const ConvParams p) {
    constexpr int TILE = C1_TILE / CO;
    __shared__ float D[CO][C1_KMAX][TILE + C1_KMAX];     // d_k,co of the tile's input rows (row index relative to t0 - pad_l)
    __shared__ double red[64];
    const int C_in = p.C_in, K = p.K;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, b = blockIdx.y;
    const int t0 = blockIdx.x * TILE;
    const bool has1 = p.in1.x != nullptr;
    const int jchunk = lane & 7, rsub = lane >> 3;
    const int c = jchunk * 4;
    const float* x0 = p.in0.x + (long long)b * p.in0.clip_stride + (long long)p.in0.row_off * C_in;
    const float* x1 = has1 ? p.in1.x + (long long)b * p.in1.clip_stride + (long long)p.in1.row_off * C_in : nullptr;
    float4 a0 = make_float4(1.f, 1.f, 1.f, 1.f), b0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, b1 = b0;
    if (p.in0.coef) {
        const float* cf = p.in0.coef + (long long)b * 2 * C_in;
        a0 = __ldg(reinterpret_cast<const float4*>(cf + c)); b0 = __ldg(reinterpret_cast<const float4*>(cf + C_in + c));
    }
    if (has1 && p.in1.coef) {
        const float* cf = p.in1.coef + (long long)b * 2 * C_in;
        a1 = __ldg(reinterpret_cast<const float4*>(cf + c)); b1 = __ldg(reinterpret_cast<const float4*>(cf + C_in + c));
    }
    float4 w[C1_KMAX][CO];                               // w[k][co] = taps of channels c..c+3 (packed [k][ci][co])
#pragma unroll
    for (int k = 0; k < C1_KMAX; ++k) {
        if (CO == 1) {
            w[k][0] = k < K ? __ldg(reinterpret_cast<const float4*>(p.w + k * C_in + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
            float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo;   // (c, co0) (c, co1) (c+1, co0) (c+1, co1) | c+2, c+3
            if (k < K) {
                lo = __ldg(reinterpret_cast<const float4*>(p.w + (k * C_in + c) * CO));
                hi = __ldg(reinterpret_cast<const float4*>(p.w + (k * C_in + c) * CO + 4));
            }
            w[k][0] = make_float4(lo.x, lo.z, hi.x, hi.z);
            w[k][CO - 1] = make_float4(lo.y, lo.w, hi.y, hi.w);
        }
    }
    const int gt_max = (p.T_out - 1) - p.pad_l + (K - 1);
    const int R = min(TILE, p.T_out - t0) + K - 1;      // input rows of this tile
    constexpr int UNR = 4;                               // rows in flight per lane
    for (int rbase = warp * 4; rbase < R; rbase += 8 * 4 * UNR) {      // warp-uniform trip count (full-mask shuffles inside)
        const int r0 = rbase + rsub;
        float4 xv[UNR], yv[UNR];
        bool ok[UNR];
#pragma unroll
        for (int i = 0; i < UNR; ++i) {
            const int row = r0 + i * 32;
            const int gt = t0 - p.pad_l + row;
            const int src = reflect_index(gt, p.T_ext);
            ok[i] = row < R && gt <= gt_max && src >= 0 && src < p.T_in;
            xv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            yv[i] = xv[i];
            if (ok[i]) {
                const long long off = (long long)src * C_in + c;
                xv[i] = __ldcs(reinterpret_cast<const float4*>(x0 + off));
                if (has1) yv[i] = __ldcs(reinterpret_cast<const float4*>(x1 + off));
            }
        }
#pragma unroll
        for (int i = 0; i < UNR; ++i) {
            const int row = r0 + i * 32;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ok[i]) {
                v.x = fmaf(xv[i].x, a0.x, b0.x); v.y = fmaf(xv[i].y, a0.y, b0.y); v.z = fmaf(xv[i].z, a0.z, b0.z); v.w = fmaf(xv[i].w, a0.w, b0.w);
                if (has1) {
                    v.x = v.x + fmaf(yv[i].x, a1.x, b1.x); v.y = v.y + fmaf(yv[i].y, a1.y, b1.y);
                    v.z = v.z + fmaf(yv[i].z, a1.z, b1.z); v.w = v.w + fmaf(yv[i].w, a1.w, b1.w);
                }
                if (p.elu) { v.x = elu1(v.x); v.y = elu1(v.y); v.z = elu1(v.z); v.w = elu1(v.w); }
            }
            float mine[CO];
#pragma unroll
            for (int co = 0; co < CO; ++co) mine[co] = 0.f;
#pragma unroll
            for (int k = 0; k < C1_KMAX; ++k) {
#pragma unroll
                for (int co = 0; co < CO; ++co) {
                    const float4 wk = w[k][co];
                    float d = fmaf(v.w, wk.w, fmaf(v.z, wk.z, fmaf(v.y, wk.y, v.x * wk.x)));
                    d += __shfl_xor_sync(0xffffffffu, d, 1);
                    d += __shfl_xor_sync(0xffffffffu, d, 2);
                    d += __shfl_xor_sync(0xffffffffu, d, 4);
                    if (jchunk == k) mine[co] = d;
                }
            }
            if (row < R && jchunk < K) {
#pragma unroll
                for (int co = 0; co < CO; ++co) D[co][jchunk][row] = mine[co];
            }
        }
    }
    __syncthreads();
    float bias[CO];
#pragma unroll
    for (int co = 0; co < CO; ++co) bias[co] = __ldg(p.bias + co);
    float s = 0.f, ss = 0.f;
    float* outb = p.out + (long long)b * p.out_clip_stride;
#pragma unroll
    for (int i = 0; i < TILE / C1_THREADS; ++i) {
        const int tl = tid + C1_THREADS * i, t = t0 + tl;
        if (t < p.T_out) {
            float o[CO];
#pragma unroll
            for (int co = 0; co < CO; ++co) {
                float acc = 0.f;
                for (int k = 0; k < K; ++k) acc += D[co][k][tl + k];
                o[co] = acc + bias[co];
                s += o[co]; ss = fmaf(o[co], o[co], ss);
            }
            if (CO == 1) outb[t] = o[0];
            else *reinterpret_cast<float2*>(outb + (long long)t * CO) = make_float2(o[0], o[CO - 1]);
        }
    }
    if (p.partials) {
        double ds = (double)s, dss = (double)ss;
        block_reduce_2d(ds, dss, red);
        if (tid == 0) {
            double* dst = p.partials + ((long long)b * gridDim.x + blockIdx.x) * 2;
            dst[0] = ds; dst[1] = dss;
        }
    }
}

bool conv_cout1_supported(const ConvParams& p) {
    return (p.C_out == 1 || p.C_out == 2) && p.S == 1 && p.D == 1 && !p.pad_zero && !p.div_scale && !p.in_ch_stride &&
           p.C_in == 32 && p.K <= C1_KMAX && !(p.in0.stats && !p.in0.coef) && !(p.in1.x && p.in1.stats && !p.in1.coef);
}
int conv_cout1_num_parts(int T_out, int C_out) {
    const int tile = C1_TILE / C_out;
    return (T_out + tile - 1) / tile;
}

cudaError_t launch_conv_cout1(const ConvParams& p, int B, cudaStream_t st, int* nparts) {
    dim3 grid(conv_cout1_num_parts(p.T_out, p.C_out), B);
    *nparts = grid.x;
    if (p.C_out == 2) conv1d_cout1_kernel<2><<<grid, C1_THREADS, 0, st>>>(p);
    else conv1d_cout1_kernel<1><<<grid, C1_THREADS, 0, st>>>(p);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------ host side
static size_t conv_smem_bytes(const ConvParams& p, int T_TILE, int CO_TILE) {
    const int R = (T_TILE - 1) * p.S + (p.K - 1) * p.D + 1;
    size_t coef = (size_t)p.C_in * (p.in1.x ? 4 : 2) + 4;
    return (coef + (size_t)p.K * p.cic * CO_TILE + (size_t)R * (p.cic + 1)) * sizeof(float);
}

template <int TX, int TM, bool TWO>
static cudaError_t launch_cfg(ConvParams p, int B, cudaStream_t st, int* nparts_out) {
    constexpr int CO_TILE = TX * 8, T_TILE = (256 / TX) * TM;
    // largest power-of-two channel chunk that fits the shared-memory budget
    const size_t budget = TWO ? 160 * 1024 : 100 * 1024;
    int cic = 32;
    while (cic > 1 && (p.C_in % cic != 0)) cic >>= 1;
    p.cic = cic;
    while (p.cic > 1 && conv_smem_bytes(p, T_TILE, CO_TILE) > budget) p.cic >>= 1;
    const size_t smem = conv_smem_bytes(p, T_TILE, CO_TILE);
    if (smem > 220 * 1024) return cudaErrorInvalidConfiguration;
    auto kern = conv1d_cl_kernel<TX, TM, TWO>;
    {
        cudaError_t e = ensure_dynamic_smem((const void*)kern, 220 * 1024);
        if (e != cudaSuccess) return e;
    }
    dim3 grid((p.T_out + T_TILE - 1) / T_TILE, (p.C_out + CO_TILE - 1) / CO_TILE, B);
    *nparts_out = grid.x * grid.y;
    kern<<<grid, 256, smem, st>>>(p);
    return cudaGetLastError();
}

int conv_num_parts(int T_out, int C_out, int C_in, int K, int B) {
    int tx, tm; bool two;
    conv_pick_tile(T_out, C_out, C_in, K, B, &tx, &tm, &two);
    const int CO_TILE = tx * 8, T_TILE = (256 / tx) * tm;
    return ((T_out + T_TILE - 1) / T_TILE) * ((C_out + CO_TILE - 1) / CO_TILE);
}

void conv_pick_tile(int T_out, int C_out, int C_in, int K, int B, int* tx, int* tm, bool* two) {
    *tx = C_out >= 128 ? 16 : (C_out >= 64 ? 8 : (C_out >= 32 ? 4 : 2));
    *two = (long long)C_in * K >= 1024;
    *tm = 8;
    // small problems: halve the time tile so that the grid covers the 148 SMs
    const int CO_TILE = *tx * 8, T_TILE = (256 / *tx) * 8;
    const long long ctas = (long long)((T_out + T_TILE - 1) / T_TILE) * ((C_out + CO_TILE - 1) / CO_TILE) * B;
    if (ctas < 2 * 148) *tm = 4;
}

cudaError_t launch_conv(const ConvParams& p, int B, cudaStream_t st, int* nparts) {
    int tx, tm; bool two;
    conv_pick_tile(p.T_out, p.C_out, p.C_in, p.K, B, &tx, &tm, &two);
#define FCB_CASE(TX_, TM_, TWO_) if (tx == TX_ && tm == TM_ && two == TWO_) return launch_cfg<TX_, TM_, TWO_>(p, B, st, nparts);
    FCB_CASE(2, 8, false) FCB_CASE(2, 4, false) FCB_CASE(4, 8, false) FCB_CASE(4, 4, false)
    FCB_CASE(8, 8, false) FCB_CASE(8, 4, false) FCB_CASE(16, 8, false) FCB_CASE(16, 4, false)
    FCB_CASE(2, 8, true) FCB_CASE(2, 4, true) FCB_CASE(4, 8, true) FCB_CASE(4, 4, true)
    FCB_CASE(8, 8, true) FCB_CASE(8, 4, true) FCB_CASE(16, 8, true) FCB_CASE(16, 4, true)
#undef FCB_CASE
    return cudaErrorInvalidConfiguration;
}

cudaError_t launch_stats_finalize(const double* partials, int nparts, double count, float eps, int mode,
                                  float* out, int B, cudaStream_t st, const float* gamma, const float* beta, int C,
                                  float* coef) {
    stats_finalize_kernel<<<B, 256, 0, st>>>(partials, nparts, count, eps, mode, out, gamma, beta, C, coef);
    return cudaGetLastError();
}

cudaError_t launch_sumsq_partials(const float* x, int B, int L, double* partials, int* nparts, cudaStream_t st, int C) {
    const int chunk = 16384;
    const int n = (L + chunk - 1) / chunk;
    *nparts = n;
    if (C == 2) sumsq_partials_kernel<2><<<dim3(n, B), 256, 0, st>>>(x, L, chunk, partials);
    else sumsq_partials_kernel<1><<<dim3(n, B), 256, 0, st>>>(x, L, chunk, partials);
    return cudaGetLastError();
}

int sumsq_num_parts(int L) { return (L + 16383) / 16384; }

}  // namespace fcb
