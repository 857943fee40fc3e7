// Small elementwise kernels around the stacks.
#include "common.cuh"
#include "kernels.h"

#include <map>
#include <mutex>
#include <utility>

namespace fcb {

cudaError_t ensure_dynamic_smem(const void* kernel, int bytes) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, int> done;     // (kernel, device) -> bytes granted
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    auto key = std::make_pair(kernel, dev);
    auto it = done.find(key);
    if (it != done.end() && it->second >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done[key] = bytes;
    return e;
}

// Final GroupNorm(1, C) of the decoder's last conv (seanet_decoder.py:160-164 -> conv.py:162), optional
// `out * scale` (codec_basic.py:405-407) and the `[:, :, :L]` trim (codec_basic.py:711) in one pass.  The raw conv output is
// channels-last [B][T_raw][C]; the waveform is written channel-planar [B][C][out_len] (C = 2: stereo, one scale per clip).
template <int C>
__global__ void final_output_kernel(const float* __restrict__ raw, const float* __restrict__ stats,
                                    const float* __restrict__ gamma, const float* __restrict__ beta,
                                    const float* __restrict__ scale, int T_raw, int out_len, float* __restrict__ out) {
    const int b = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= out_len) return;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        float v = raw[((long long)b * T_raw + t) * C + c];
        if (stats) {   // deferred GroupNorm(1, C) of the last conv (norm: time_group_norm); weight_norm / none output is plain
            const float mean = stats[2 * b], rstd = stats[2 * b + 1];
            const float a = rstd * gamma[c];
            v = fmaf(v, a, beta[c] - a * mean);
        }
        if (scale) v = v * scale[b];
        out[((long long)b * C + c) * out_len + t] = v;
    }
}

__global__ void fill_kernel(float* p, float v, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

cudaError_t launch_final_output(const float* raw, const float* stats, const float* gamma, const float* beta,
                                const float* scale, int B, int T_raw, int out_len, float* out, cudaStream_t st, int C) {
    if (C == 2)
        final_output_kernel<2><<<dim3((out_len + 255) / 256, B), 256, 0, st>>>(raw, stats, gamma, beta, scale, T_raw, out_len, out);
    else
        final_output_kernel<1><<<dim3((out_len + 255) / 256, B), 256, 0, st>>>(raw, stats, gamma, beta, scale, T_raw, out_len, out);
    return cudaGetLastError();
}

// ---- segment_dur != None (Encodec._encode / _decode, codec_basic.py:334-359,382-396)
// A planar multi-channel batch [B][C][L] is passed as B*C single-channel rows: the gathered segments are then
// [(s*B + b)][C][seg_len], and the overlap-add applies the same triangular weights to every channel (codec_basic.py:77-116).
// Segments as a batch: out[(s*B + b)][j] = wav[b][(s0 + s)*stride + j], j < seg_len (every gathered segment is full length).
__global__ void gather_segments_kernel(const float* __restrict__ wav, int B, int L, int seg_len, int stride, int s0,
                                       float* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y, s = blockIdx.z;
    if (j >= seg_len) return;
    out[((long long)s * B + b) * seg_len + j] = wav[(long long)b * L + (long long)(s0 + s) * stride + j];
}

cudaError_t launch_gather_segments(const float* wav, int B, int L, int seg_len, int stride, int s0, int n_seg, float* out,
                                   cudaStream_t st) {
    if (n_seg <= 0) return cudaSuccess;
    gather_segments_kernel<<<dim3((seg_len + 255) / 256, B, n_seg), 256, 0, st>>>(wav, B, L, seg_len, stride, s0, out);
    return cudaGetLastError();
}

// _linear_overlap_add (codec_basic.py:77-116): out[n] = sum_i w[n - i*stride] * frame_i[n - i*stride] / sum_i w[n - i*stride],
// frames in ascending order like the reference's running sums; w = 0.5 - |t - 0.5| with t = linspace(0, 1, dl0 + 2)[1:-1]
// taken from the FIRST frame's length (ATen's linspace: start + step*k below the midpoint, end - step*(steps-1-k) above).
__global__ void overlap_add_kernel(const OlaParams p) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (n >= p.out_len) return;
    const int steps = p.dl0 + 2;
    const float step = 1.0f / (float)(steps - 1);
    const int halfway = steps / 2;
    int i_lo = 0;
    if (n >= p.dl0) i_lo = (n - p.dl0) / p.stride + 1;
    int i_hi = n / p.stride;
    if (i_hi > p.n_seg - 1) i_hi = p.n_seg - 1;
    float acc = 0.f, sw = 0.f;
    for (int i = i_lo; i <= i_hi; ++i) {
        const int j = n - i * p.stride;
        const float* fr;
        int dl;
        if (i < p.n_full) { dl = p.dl0; fr = p.full + ((long long)i * p.B + b) * p.dl0; }
        else { dl = p.tail_dl[i - p.n_full]; fr = p.tail[i - p.n_full] + (long long)b * dl; }
        if (j >= dl) continue;
        const int k = j + 1;
        const float t = k < halfway ? step * (float)k : 1.0f - step * (float)(steps - k - 1);
        const float w = 0.5f - fabsf(t - 0.5f);
        acc = __fadd_rn(acc, __fmul_rn(w, fr[j]));
        sw = __fadd_rn(sw, w);
    }
    p.out[(long long)b * p.out_len + n] = acc / sw;
}

cudaError_t launch_overlap_add(const OlaParams& p, cudaStream_t st) {
    overlap_add_kernel<<<dim3((p.out_len + 255) / 256, p.B), 256, 0, st>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_fill(float* p, float v, long long n, cudaStream_t st) {
    fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p, v, n);
    return cudaGetLastError();
}

}  // namespace fcb
