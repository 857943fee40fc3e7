// SLSTM recurrence as ONE persistent cooperative kernel per layer (fp32 SIMT).
// Reference: funcodec/modules/normed_modules/lstm.py:12-28 (nn.LSTM(dim, dim, num_layers), gate order
// i,f,g,o, zero initial state, y = lstm(x) + x).
//
// The input projections x_t W_ih^T + b_ih + b_hh for all t are one GEMM (conv kernel as a 1x1 conv) written
// as gx[B][T][4H] with unit-major packed columns (n' = 4*j + gate).  The recurrence
//     gates = gx[:, t] + h_{t-1} W_hh^T ;  c = sig(f) c + sig(i) tanh(g) ;  h = sig(o) tanh(c)
// is strictly sequential in t, so the kernel is built around latency:
//   * grid = H / UNITS CTAs (<= 148, one per SM, cooperative launch), CTA j owns hidden units
//     [j*UNITS, (j+1)*UNITS) and keeps its W_hh slice [H][4*UNITS] (128 KB at H=1024) in shared memory for
//     all T steps -- W_hh is read from HBM/L2 exactly once per layer instead of once per step;
//   * per step every CTA needs the whole h_{t-1} of a clip group: it is exchanged through global memory (L2)
//     with a per-group release/acquire counter barrier; independent clip groups (8 clips) are software
//     pipelined so that one group's barrier + broadcast latency hides behind the other group's math;
//   * a thread accumulates the 4 gates of one unit for 8 clips (32 fp32 accumulators) over an interleaved
//     K slice (W rows via conflict-free LDS.128, h via broadcast LDS.128), K slices are reduced with
//     shuffles + one shared-memory pass, and UNITS*8 threads do the cell update.
// Latency-bound by construction (T' dependent steps); FLOPs = 2*B*T*4H*H per layer.
#include <cooperative_groups.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "kernels.h"
#include "tc_sm100.cuh"

namespace fcb {

// clips per work item (accumulator tile).  4-clip groups (4 independent chains for B = 16) were measured twice: on the 2-slot
// ring of round 1 (no gain) and with one ring slot per group (r2d: 3.67 vs 3.32 ms per SLSTM at config 2) -- the per-item
// fixed costs (poll, bulk copy, reduction, publish) outweigh the shorter gate GEMM.
constexpr int LSTM_GB = 8;
constexpr int LSTM_NBUF_MAX = 8;  // h ring depth: 2 .. 8 slots, as many as shared memory holds (more independent clip groups in flight)
constexpr int LSTM_THREADS = 480; // 8 compute warps, up to 3 x 2 cell warps (items round-robin), 1 loader warp: 15 warps keep the
                                  // 128-register budget of the 16-warp allocation bucket (17 warps drop to 96: measured slower)
constexpr int LSTM_PAIRS_MAX = 3;
constexpr int LSTM_MAX_GROUPS = 64;

// Gates on the hardware ex2 / rcp units: ~3e-7 relative instead of ~1e-7 for expf / tanhf, a much shorter dependent chain in
// the cell phase that heads every timestep's critical path.  Measured (r2fc): 17.73 -> 17.44 ms per config-2 step with an
// IDENTICAL parity table (same 3999 / 4000 frames, waveforms 1.2e-6).
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sigmoid_fast(float x) { return rcp_approx(1.0f + tc::exp2f_approx(-1.4426950408889634f * x)); }
__device__ __forceinline__ float tanh_fast(float x) { return fmaf(-2.0f, rcp_approx(1.0f + tc::exp2f_approx(2.8853900817779268f * x)), 1.0f); }

__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// PROFILING ONLY: CTA 0 stamps event e of work item i (items of the steps from LSTM_TRACE_FIRST_STEP on)
#define LSTM_TRACE(i, e)                                                                             \
    do {                                                                                             \
        if (p.trace && blockIdx.x == 0) {                                                            \
            const int ti__ = (i) - LSTM_TRACE_FIRST_STEP * ng;                                       \
            if (ti__ >= 0 && ti__ < LSTM_TRACE_ITEMS) p.trace[ti__ * 8 + (e)] = gtimer();            \
        }                                                                                            \
    } while (0)

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Work item (t, g) = timestep t of clip group g (8 clips).  Clip groups are independent sequences and each has
// its own release/acquire counter, so the kernel is warp-specialised around items instead of CTA-wide barriers:
//   * loader warp (1 lane): waits for a free h ring slot, polls the group's counter until every CTA has published
//     h_{t-1}, then pulls the 8 rows [H] straight from L2 into shared memory with cp.async.bulk (mbarrier tx);
//   * 8 compute warps: wait for the slot, accumulate gates = h_{t-1} W_hh^T for the CTA's 4*UNITS columns (K split
//     over warps/lanes, shuffle-reduced), drop the partials in a double-buffered exchange area;
//   * 2 x 2 cell warps (alternate items): add the partials and gx (prefetched one item ahead), run the cell update,
//     store h_t (+ skip output) and publish the group's counter with a single release-add.
// The barrier/broadcast latency of one group is hidden behind the math of the others; with a single group
// (B <= 8) the chain is latency-bound by construction.
// mma.sync m16n8k16 (fp16 operands, fp32 accumulate): D += A * B, A = 16 gate columns x 16 k (row-major fragments), B = 16 k x 8 clips
__device__ __forceinline__ void mma_16816(float (&c)[4], const uint4& a, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b0), "r"(b1));
}
constexpr float LSTM_H_SCALE = 4096.0f;   // |h| < 1: fp16 operand scale of the hidden state (power of two)

// MMA = true: the gate GEMM h_{t-1} W_hh^T of an item runs on the tensor cores (mma.sync m16n8k16, N = the 8 clips of the group)
// with the 3-term FP16 split of conv_tc.cu (W pre-scaled per layer so that max|w| is in [2^13, 2^14), h scaled by 2^12;
// lo*hi + hi*lo + hi*hi in fp32, exact inverse scale afterwards): ~2^-22 relative like the fp32 FMA chain it replaces, at a
// third of the shared-memory instruction count -- the item then costs one pass over the 128 KB W_hh slice (LDS-bound).
// The W slice lives in shared memory in FRAGMENT ORDER: [k-step (16 k)][m-tile (16 columns)][hi | lo][lane][8 halfs].
template <int UNITS, bool MMA>
__global__ void __launch_bounds__(LSTM_THREADS, 1) lstm_seq_kernel(const LstmSeqParams p, const int nbuf, const int npair, const int pload, const int nset) {
    constexpr int GB = LSTM_GB;
    constexpr int COLS = 4 * UNITS;            // gate columns owned by this CTA
    constexpr int KS_PER_WARP = 32 / UNITS;    // K slices inside a warp
    // compute-warp sets: nset = 1: all 8 warps split the K dimension of one item; nset = 2 (narrow layers, where an item is bound
    // by latencies, not FMAs): two sets of 4 warps work on two consecutive items at the same time
    const int WS = 8 / nset;                   // warps per set
    const int NSLICE = WS * KS_PER_WARP;       // K slices per item (interleaved in groups of 4 k)
    constexpr int NFIN = GB * UNITS;      // active cell threads
    extern __shared__ __align__(128) float smem[];
    const int H = p.H, T = p.T, B = p.B;
    float* Ws = smem;                                   // [H][COLS]
    float* Hs = Ws + (size_t)H * COLS;                  // [nbuf][GB][H]
    float* red = Hs + nbuf * GB * H;               // [npair][8 warps][GB][COLS]
    float* cS = red + npair * 8 * GB * COLS;       // [ng][GB][UNITS] cell state
    const int ng = (B + GB - 1) / GB;
    uint64_t* bars = reinterpret_cast<uint64_t*>(cS + ((ng * GB * UNITS + 3) & ~3));
    uint64_t* hs_full = bars;                           // [nbuf] tx
    uint64_t* hs_empty = hs_full + nbuf;                // [nbuf] 8 compute-warp arrivals
    uint64_t* red_full = hs_empty + nbuf;               // [npair] 8 compute-warp arrivals
    uint64_t* red_empty = red_full + LSTM_PAIRS_MAX;    // [npair] 64 cell-thread arrivals
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int j0 = blockIdx.x * UNITS;
    const int n_items = T * ng;
    const unsigned nctas = gridDim.x;

    // W_hh slice in the FFMA2-friendly layout: for every pair of consecutive k and every unit u two 16-byte records
    //   rec(kp, half, u) = { W[k][u][2*half], W[k+1][u][2*half], W[k][u][2*half+1], W[k+1][u][2*half+1] }
    // so that one LDS.128 yields two (w_k, w_{k+1}) register pairs and lanes u = 0..UNITS-1 read consecutive records.
    if (MMA) {
        constexpr int MT = COLS / 16;
        __half* Wf = reinterpret_cast<__half*>(Ws);
        for (int e = tid; e < H * COLS; e += LSTM_THREADS) {
            const int k = e / COLS, c = e - k * COLS;
            const float v = __ldg(p.whh + (long long)k * 4 * H + (long long)j0 * 4 + c) * p.whh_scale;
            const __half vh = __float2half_rn(v);
            const __half vl = __float2half_rn(v - __half2float(vh));
            const int ksg = k >> 4, kk = k & 15, mt = c >> 4, r = c & 15;
            const int ln = (r & 7) * 4 + ((kk & 7) >> 1);
            const int hidx = (kk >= 8 ? 4 : 0) + (r >= 8 ? 2 : 0) + (kk & 1);
            const size_t base = ((size_t)(ksg * MT + mt) * 2 * 32 + ln) * 8 + hidx;
            Wf[base] = vh;
            Wf[base + 32 * 8] = vl;
        }
    } else
    for (int e = tid; e < H * COLS; e += LSTM_THREADS) {
        const int k = e / COLS, c = e - k * COLS;
        const int uu = c >> 2, g = c & 3;
        const int dst = (((k >> 1) * 2 + (g >> 1)) * UNITS + uu) * 4 + ((g & 1) * 2 + (k & 1));
        Ws[dst] = __ldg(p.whh + (long long)k * 4 * H + (long long)j0 * 4 + c);
    }
    for (int e = tid; e < ng * GB * UNITS; e += LSTM_THREADS) cS[e] = 0.f;
    if (tid == 0) {
        for (int i = 0; i < nbuf; ++i) { tc::mbar_init(hs_full + i, 1); tc::mbar_init(hs_empty + i, WS); }
        for (int i = 0; i < LSTM_PAIRS_MAX; ++i) { tc::mbar_init(red_full + i, WS); tc::mbar_init(red_empty + i, 64); }
        tc::mbar_fence_init();
    }
    __syncthreads();

    if (warp < 8) {
        // ================================================================ compute warps
        const int u = lane % UNITS, ks = lane / UNITS;
        const int set = warp / WS, wset = warp - set * WS;
        const int slice = wset * KS_PER_WARP + ks;
        for (int i = ng + set; i < n_items; i += nset) {        // items with t == 0 need no recurrent term
            const int n = i - ng;
            const int hb = n % nbuf, rb = n % npair;
            tc::mbar_wait(hs_full + hb, (uint32_t)((n / nbuf) & 1));
            if (tid == 0) LSTM_TRACE(i, 2);
            const float* Hc = Hs + hb * GB * H;
            if (MMA) {
                constexpr int MT = COLS / 16;
                constexpr int KSW_MAX = 8;                              // k-steps per warp (host guarantees ksw <= 8)
                const int g8 = lane >> 2, t4 = lane & 3;
                const int ksw = (H >> 4) / WS;                          // k-steps of this warp
                const uint4* Wf = reinterpret_cast<const uint4*>(Ws);
                // B fragments of this lane (clip g8, k pairs) from the staged h_{t-1} rows
                const float* hrow = Hc + g8 * H + wset * ksw * 16 + t4 * 2;
                float2 xs[2 * KSW_MAX];
#pragma unroll
                for (int j = 0; j < KSW_MAX; ++j) {
                    xs[2 * j] = make_float2(0.f, 0.f);
                    xs[2 * j + 1] = make_float2(0.f, 0.f);
                    if (j < ksw) {
                        xs[2 * j] = *reinterpret_cast<const float2*>(hrow + j * 16);
                        xs[2 * j + 1] = *reinterpret_cast<const float2*>(hrow + j * 16 + 8);
                    }
                }
                // three independent accumulator chains per m-tile (hi*hi, lo*hi, hi*lo), summed at the end: the dependent-MMA chain
                // is ksw long instead of 3 * ksw
                float c[MT][3][4];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                    for (int q = 0; q < 3; ++q) { c[mt][q][0] = 0.f; c[mt][q][1] = 0.f; c[mt][q][2] = 0.f; c[mt][q][3] = 0.f; }
#pragma unroll
                for (int j = 0; j < KSW_MAX; ++j) {
                    if (j < ksw) {
                        const int ksg = wset * ksw + j;
                        uint32_t bh0, bl0, bh1, bl1;
                        tc::split_f16x2(xs[2 * j].x * LSTM_H_SCALE, xs[2 * j].y * LSTM_H_SCALE, bh0, bl0);
                        tc::split_f16x2(xs[2 * j + 1].x * LSTM_H_SCALE, xs[2 * j + 1].y * LSTM_H_SCALE, bh1, bl1);
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) {
                            const uint4 ah = Wf[((size_t)(ksg * MT + mt) * 2 + 0) * 32 + lane];
                            const uint4 al = Wf[((size_t)(ksg * MT + mt) * 2 + 1) * 32 + lane];
                            mma_16816(c[mt][0], ah, bh0, bh1);
                            mma_16816(c[mt][1], al, bh0, bh1);
                            mma_16816(c[mt][2], ah, bl0, bl1);
                        }
                    }
                }
                __syncwarp();
                if (tid == 0) LSTM_TRACE(i, 3);
                if (lane == 0) tc::mbar_arrive(hs_empty + hb);       // this warp is done with the h slot
                tc::mbar_wait(red_empty + rb, (uint32_t)((n / npair) & 1) ^ 1);
                {
                    // C fragment: rows (gate columns) g8, g8 + 8 of the m-tile; columns (clips) 2*t4, 2*t4 + 1
                    const float inv = p.whh_inv_scale;
                    float* rd = red + (size_t)rb * 8 * GB * COLS + (size_t)(wset * GB + t4 * 2) * COLS + g8;
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) {
                        rd[mt * 16] = ((c[mt][1][0] + c[mt][2][0]) + c[mt][0][0]) * inv;
                        rd[COLS + mt * 16] = ((c[mt][1][1] + c[mt][2][1]) + c[mt][0][1]) * inv;
                        rd[mt * 16 + 8] = ((c[mt][1][2] + c[mt][2][2]) + c[mt][0][2]) * inv;
                        rd[COLS + mt * 16 + 8] = ((c[mt][1][3] + c[mt][2][3]) + c[mt][0][3]) * inv;
                    }
                }
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(red_full + rb);
                if (tid == 0) LSTM_TRACE(i, 4);
                continue;
            }
            // packed fp32 FMAs (FFMA2): even-k and odd-k partial sums live in the two halves of a register pair
            float2 acc2[4][GB];
#pragma unroll
            for (int gg = 0; gg < 4; ++gg)
#pragma unroll
                for (int bb = 0; bb < GB; ++bb) acc2[gg][bb] = make_float2(0.f, 0.f);
            for (int k0 = slice * 4; k0 < H; k0 += NSLICE * 4) {
                const int kp = k0 >> 1;
                const float4 wa0 = *reinterpret_cast<const float4*>(Ws + (((kp + 0) * 2 + 0) * UNITS + u) * 4);
                const float4 wb0 = *reinterpret_cast<const float4*>(Ws + (((kp + 0) * 2 + 1) * UNITS + u) * 4);
                const float4 wa1 = *reinterpret_cast<const float4*>(Ws + (((kp + 1) * 2 + 0) * UNITS + u) * 4);
                const float4 wb1 = *reinterpret_cast<const float4*>(Ws + (((kp + 1) * 2 + 1) * UNITS + u) * 4);
#pragma unroll
                for (int bb = 0; bb < GB; ++bb) {
                    const float4 h4 = *reinterpret_cast<const float4*>(Hc + bb * H + k0);
                    const float2 h01 = make_float2(h4.x, h4.y), h23 = make_float2(h4.z, h4.w);
                    acc2[0][bb] = __ffma2_rn(h01, make_float2(wa0.x, wa0.y), acc2[0][bb]);
                    acc2[1][bb] = __ffma2_rn(h01, make_float2(wa0.z, wa0.w), acc2[1][bb]);
                    acc2[2][bb] = __ffma2_rn(h01, make_float2(wb0.x, wb0.y), acc2[2][bb]);
                    acc2[3][bb] = __ffma2_rn(h01, make_float2(wb0.z, wb0.w), acc2[3][bb]);
                    acc2[0][bb] = __ffma2_rn(h23, make_float2(wa1.x, wa1.y), acc2[0][bb]);
                    acc2[1][bb] = __ffma2_rn(h23, make_float2(wa1.z, wa1.w), acc2[1][bb]);
                    acc2[2][bb] = __ffma2_rn(h23, make_float2(wb1.x, wb1.y), acc2[2][bb]);
                    acc2[3][bb] = __ffma2_rn(h23, make_float2(wb1.z, wb1.w), acc2[3][bb]);
                }
            }
            float acc[4][GB];
#pragma unroll
            for (int gg = 0; gg < 4; ++gg)
#pragma unroll
                for (int bb = 0; bb < GB; ++bb) acc[gg][bb] = acc2[gg][bb].x + acc2[gg][bb].y;
            __syncwarp();
            if (tid == 0) LSTM_TRACE(i, 3);
            if (lane == 0) tc::mbar_arrive(hs_empty + hb);           // this warp is done with the h slot
#pragma unroll
            for (int gg = 0; gg < 4; ++gg)
#pragma unroll
                for (int bb = 0; bb < GB; ++bb) {
                    float v = acc[gg][bb];
#pragma unroll
                    for (int o = UNITS; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                    acc[gg][bb] = v;
                }
            tc::mbar_wait(red_empty + rb, (uint32_t)((n / npair) & 1) ^ 1);
            if (ks == 0) {
                float* rd = red + (size_t)rb * 8 * GB * COLS;
#pragma unroll
                for (int bb = 0; bb < GB; ++bb)
                    *reinterpret_cast<float4*>(rd + (wset * GB + bb) * COLS + u * 4) =
                        make_float4(acc[0][bb], acc[1][bb], acc[2][bb], acc[3][bb]);
            }
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(red_full + rb);
            if (tid == 0) LSTM_TRACE(i, 4);
        }
    } else if (warp < 8 + 2 * LSTM_PAIRS_MAX) {
        // ================================================================ cell warps: npair pairs take the items round-robin
        const int pair = (warp - 8) >> 1;
        if (pair >= npair) return;
        const int ftid = (tid - 256) & 63;
        const int fbb = ftid / UNITS, fu = ftid % UNITS;
        const bool active = ftid < NFIN;
        auto load_gx = [&](int i) -> float4 {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < n_items) {
                const int t = i / ng, g = i - t * ng;
                const int b0 = g * GB;
                if (active && b0 + fbb < B)
                    v = __ldcs(reinterpret_cast<const float4*>(p.gx + ((long long)(b0 + fbb) * T + t) * 4 * H + (long long)(j0 + fu) * 4));
            }
            return v;
        };
        auto load_skip = [&](int i) -> float {       // raw SLSTM input of this thread's (clip, unit) for item i (last layer only)
            float v = 0.f;
            if (p.y_out && i < n_items) {
                const int t = i / ng, g = i - t * ng;
                const int b = g * GB + fbb;
                if (active && b < B) v = __ldcs(p.skip.x + (long long)b * p.skip.clip_stride + ((long long)(p.skip.row_off + t)) * H + j0 + fu);
            }
            return v;
        };
        // items of this pair: those whose exchange buffer (i - ng) % npair == pair; the t == 0 items (i < ng) use no buffer and are
        // spread the same way
        const int first = (pair + ng) % npair;                        // smallest i >= 0 with (i - ng) % npair == pair
        float4 gxv = load_gx(first);
        float skv = load_skip(first);
        for (int i = first; i < n_items; i += npair) {
            const int t = i / ng, g = i - t * ng;
            const int b0 = g * GB;
            const int nb = min(GB, B - b0);
            const bool mine = active && fbb < nb;
            const float4 gx_next = load_gx(i + npair);           // in flight while this item is reduced
            const float sk_next = load_skip(i + npair);
            float g4[4] = {gxv.x, gxv.y, gxv.z, gxv.w};
            if (t > 0) {
                const int n = i - ng, rb = pair;                 // == n % npair by construction
                tc::mbar_wait_backoff(red_full + rb, (uint32_t)((n / npair) & 1), 64);
                if (ftid == 0) LSTM_TRACE(i, 5);
                if (mine) {
                    const float* rd = red + (size_t)rb * 8 * GB * COLS;
                    float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int w8 = 0; w8 < WS; ++w8) {
                        const float4 r4 = *reinterpret_cast<const float4*>(rd + (w8 * GB + fbb) * COLS + fu * 4);
                        s4.x += r4.x; s4.y += r4.y; s4.z += r4.z; s4.w += r4.w;
                    }
                    g4[0] += s4.x; g4[1] += s4.y; g4[2] += s4.z; g4[3] += s4.w;
                }
                tc::mbar_arrive(red_empty + rb);
            }
            float h = 0.f;
            long long o = 0;
            if (mine) {
                const int b = b0 + fbb, j = j0 + fu;
                const float ig = sigmoid_fast(g4[0]), fg = sigmoid_fast(g4[1]), gg = tanh_fast(g4[2]), og = sigmoid_fast(g4[3]);
                float* cp = cS + (g * GB + fbb) * UNITS + fu;
                const float c = fg * (*cp) + ig * gg;
                *cp = c;
                h = og * tanh_fast(c);
                o = ((long long)b * T + t) * H + j;
                __stcg(p.h_seq + o, h);
            }
            // publish h_t of this group FIRST (it heads every other CTA's critical path): the pair's stores -> named barrier ->
            // one gpu-scope release add; the skip output below is off the recurrence
            asm volatile("bar.sync %0, 64;" ::"r"(3 + pair) : "memory");
            if (ftid == 0 && t + 1 < T)
                asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p.barrier + g), "r"(1u) : "memory");
            if (ftid == 0) LSTM_TRACE(i, 6);
            if (mine && p.y_out) {
                const int b = b0 + fbb, j = j0 + fu;
                float xv = skv;
                if (p.skip.stats) {
                    const float mean = p.skip.stats[2 * b], rstd = p.skip.stats[2 * b + 1];
                    const float a = rstd * p.skip.gamma[j];
                    xv = fmaf(xv, a, p.skip.beta[j] - a * mean);
                }
                p.y_out[o] = h + xv;
            }
            gxv = gx_next;
            skv = sk_next;
        }
    } else {
        // ================================================================ loader warp
        if (nbuf == ng && pload) {
            // one ring slot per clip group: lane g serves group g, so the polls and copies of a timestep's groups overlap
            if (lane < ng) {
                const int g = lane, b0 = g * GB;
                const int nb = min(GB, B - b0);
                float* dst = Hs + g * GB * H;
                for (int t = 1; t < T; ++t) {
                    tc::mbar_wait_backoff(hs_empty + g, (uint32_t)((t - 1) & 1) ^ 1, 64);
                    if (lane == 0) LSTM_TRACE(t * ng, 0);
                    unsigned seen = ld_acquire_u32(p.barrier + g);
                    while (seen < (unsigned)t * nctas) seen = ld_acquire_u32(p.barrier + g);
                    if (lane == 0) LSTM_TRACE(t * ng, 1);
                    asm volatile("fence.proxy.async;" ::: "memory");     // acquired generic writes -> visible to the bulk copy
                    tc::mbar_arrive_expect_tx(hs_full + g, (uint32_t)(nb * H * 4));
                    for (int bb = 0; bb < nb; ++bb)
                        tc::bulk_g2s(dst + bb * H, p.h_seq + ((long long)(b0 + bb) * T + (t - 1)) * H, (uint32_t)(H * 4), hs_full + g);
                }
            }
        } else if (lane == 0) {
            for (int i = ng; i < n_items; ++i) {
                const int t = i / ng, g = i - t * ng;
                const int n = i - ng, hb = n % nbuf;
                const int b0 = g * GB;
                const int nb = min(GB, B - b0);
                tc::mbar_wait_backoff(hs_empty + hb, (uint32_t)((n / nbuf) & 1) ^ 1, 64);
                LSTM_TRACE(i, 0);
                unsigned seen = ld_acquire_u32(p.barrier + g);
                while (seen < (unsigned)t * nctas) seen = ld_acquire_u32(p.barrier + g);
                LSTM_TRACE(i, 1);
                asm volatile("fence.proxy.async;" ::: "memory");     // acquired generic writes -> visible to the bulk copy
                tc::mbar_arrive_expect_tx(hs_full + hb, (uint32_t)(nb * H * 4));
                float* dst = Hs + hb * GB * H;
                for (int bb = 0; bb < nb; ++bb)
                    tc::bulk_g2s(dst + bb * H, p.h_seq + ((long long)(b0 + bb) * T + (t - 1)) * H, (uint32_t)(H * 4), hs_full + hb);
            }
        }
    }
}

size_t lstm_seq_smem_bytes(int H, int B, int units, int nbuf = 2, int npair = 2, bool ring = true) {
    constexpr int gb = LSTM_GB;
    const int ng = (B + gb - 1) / gb;
    const size_t cs = ((size_t)ng * gb * units + 3) & ~(size_t)3;
    return ((size_t)H * 4 * units + (ring ? (size_t)nbuf * gb * H : 0) + (size_t)npair * 8 * 4 * units * gb + cs) * sizeof(float) +
           (2 * nbuf + 2 * LSTM_PAIRS_MAX) * 8 + 64;
}

// h ring depth: one slot per independent clip group (their barrier / broadcast latencies overlap), 2 .. LSTM_NBUF_MAX,
// limited by shared memory (H = 1024: the 128 KB W_hh slice leaves room for 2 slots of 32 KB)
static int lstm_pick_nbuf(int H, int B, int units, bool ring) {
    const int ng = (B + LSTM_GB - 1) / LSTM_GB;
    int nbuf = ng < 2 ? 2 : (ng > LSTM_NBUF_MAX ? LSTM_NBUF_MAX : ng);
    while (nbuf > 2 && lstm_seq_smem_bytes(H, B, units, nbuf, 2, ring) > 220 * 1024) --nbuf;
    return nbuf;
}

int lstm_pick_units(int H) {
    // largest slice that fits shared memory while keeping >= 96 CTAs busy when H allows it
    if (H % 8 == 0 && lstm_seq_smem_bytes(H, 16, 8) <= 220 * 1024 && H / 8 >= 96) return 8;
    if (H % 4 == 0 && lstm_seq_smem_bytes(H, 16, 4) <= 220 * 1024) return 4;
    return 0;
}

template <int UNITS, bool MMA>
static cudaError_t launch_seq(const LstmSeqParams& p, cudaStream_t st) {
    constexpr int GB = LSTM_GB;
    int nbuf = lstm_pick_nbuf(p.H, p.B, UNITS, true);
    // cell pairs: 3 when there are at least 3 independent clip groups to keep busy and the extra exchange buffer fits
    // per-group loader lanes only pay with many groups (r2f / r2g: config 2 (2 groups) 3.7 vs 3.45 ms, config 4 (4 groups) 8.15 vs
    // 6.5 ms, config 3 (8 groups) 36.8 vs 38.0 ms per SLSTM)
    const int ngroups = (p.B + GB - 1) / GB;
    int npair = 2, pload = ngroups >= 8 ? 1 : 0;
    // two compute-warp sets when an item's gate GEMM is small (H <= 512) and there are other groups to work on
    int nset = (p.H <= 512 && ngroups >= 2) ? 2 : 1;
    if ((p.B + GB - 1) / GB >= 3 && lstm_seq_smem_bytes(p.H, p.B, UNITS, nbuf, 3) <= 220 * 1024) npair = 3;
    const size_t smem = lstm_seq_smem_bytes(p.H, p.B, UNITS, nbuf, npair);
    // the tensor-core gate GEMM needs whole k-steps per warp
    if (MMA && (p.H % 16 != 0 || ((p.H / 16) % (8 / nset)) != 0 || (p.H / 16) / (8 / nset) > 8)) return launch_seq<UNITS, false>(p, st);
    auto kern = lstm_seq_kernel<UNITS, MMA>;
    {
        cudaError_t e = ensure_dynamic_smem((const void*)kern, 225 * 1024);
        if (e != cudaSuccess) return e;
    }
    if (smem > 225 * 1024) return cudaErrorInvalidConfiguration;
    if ((p.B + GB - 1) / GB > LSTM_MAX_GROUPS) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(p.barrier, 0, LSTM_MAX_GROUPS * sizeof(unsigned), st);
    if (e != cudaSuccess) return e;
    dim3 grid(p.H / UNITS), block(LSTM_THREADS);
    LstmSeqParams pc = p;
    void* args[] = {&pc, &nbuf, &npair, &pload, &nset};
    return cudaLaunchCooperativeKernel((void*)kern, grid, block, args, smem, st);
}

cudaError_t launch_lstm_seq(const LstmSeqParams& p, cudaStream_t st) {
    if (p.H % 4 != 0) return cudaErrorInvalidValue;
    const int units = lstm_pick_units(p.H);
    const bool mma = p.whh_scale > 0.f;               // tensor-core gate GEMM; whh_scale == 0: the fp32 FFMA2 path
    if (units == 8) return mma ? launch_seq<8, true>(p, st) : launch_seq<8, false>(p, st);
    if (units == 4) return mma ? launch_seq<4, true>(p, st) : launch_seq<4, false>(p, st);
    return cudaErrorInvalidConfiguration;
}

}  // namespace fcb
