// Implicit-GEMM Conv1d on the 5th-generation tensor cores (tcgen05.mma kind::f16, accumulators in TMEM),
// fp32-faithful through a 3-term FP16 split: both operands are pre-scaled by a power of two (activations x16, weights
// per layer so that max|w| lands in [2^13, 2^14)), x = hi + lo with hi = fp16(x), lo = fp16(x - hi), and
// D += lo*hi + hi*lo + hi*hi in fp32; the epilogue multiplies by the (exact) inverse scale.  Same accuracy as the
// 3xTF32 split it replaces (both drop the lo*lo term, ~2^-22 relative), at twice the tensor throughput and half the
// shared-memory operand bytes per MAC (K = 16 per MMA instead of 8; a 128-byte swizzle row holds 64 channels).
//
// Same contract as conv_simt.cu (fused [GroupNorm apply + resblock add + ELU + reflect pad] on the input,
// bias + raw store + GroupNorm partial statistics on the output), reference semantics
// funcodec/modules/normed_modules/conv.py:243-261 / :281-305.
//
// GEMM view (channels-last makes both operands K-major):
//     D[t (M = 128 time rows), co (N = n_tile)] = sum_{tap k} sum_{ci} X[t*S + k - pad_l][ci] * W[k][ci][co]
//   * A (activations): one "unit" = (32-channel chunk, stride phase p): the rows {(t0+u)*S + p - pad_l}
//     are transformed by a producer group and written (hi and lo slabs) into the canonical SWIZZLE_128B
//     K-major layout; a ring stage holds a 64-channel chunk, i.e. two units side by side (the two producer groups
//     each fill one half; layers with a single 32-channel chunk fill half a stage and the groups alternate stages);
//     every tap k = q*S + p of that phase is then just a ROW-SHIFTED view (start address
//     + q*128 B; the hardware swizzle works on absolute address bits) of the same slab -- no im2col copy.
//   * B (weights): pre-split, pre-swizzled slab images in HBM (engine.cu pack_tc), one cp.async.bulk
//     (TMA engine, 1-D) per (chunk, tap) into a ring, completion on an mbarrier.
//   * PERSISTENT CTAs (one per SM) walk a static list of (clip, n-tile, time-tile) tiles; every role keeps
//     running across tile boundaries, so the next tile's loads overlap the previous tile's MMAs and epilogue.
//   * warp roles (22 warps): 0-7 / 8-15 two producer groups taking alternate units (two units of global
//     loads in flight; the transform is issue-bound, hence 16 warps); 16 weight copies + TMEM alloc; 17 MMA
//     issuer; 18-21 accumulator warps.
//   * the tensor core adds into its fp32 accumulator with truncation, so a TMEM-resident chain loses
//     ~1 ulp per MMA (measured 5e-5 relative after 384 chained MMAs): chains are cut every ~48 MMAs, the MMA
//     warp ping-pongs between two TMEM accumulators and the accumulator warps fold each finished group into
//     a third TMEM region (running totals) with round-to-nearest CUDA-core adds, then run the epilogue
//     (bias, channels-last store, GroupNorm partial sums) on the last group.
// Roofline: tensor pipe (3 MMAs per fp32-equivalent product) for the deep layers; HBM for the C <= 64 layers.
//
// FREQ = true is the FreqCodec 2-D mode (SConv2d / SConvTranspose2d, conv.py:317-447): a "clip" of the tile list is a
// pseudo-clip (clip b, output frequency row f_out) and the gathered input channel cg = kf*cin + c of a chunk comes from
// frequency row f_out*SF + kf - pad_f (reflect / zero indexed) of the [B][F][T][cin] input, so a 32-channel chunk holds
// 32/cin frequency taps (cin < 32) or a 32-channel slice of one tap; everything downstream of the producers (weight
// slabs [tap kt][cg][co], MMA issue, folding) is the 1-D machinery.  The epilogue scatters the phases of a transposed
// conv (co -> (pf, pt, channel)) and can store fewer channels than the padded n-tile (the 32 -> 3 output conv).
#include <cuda.h>
#include "common.cuh"
#include "kernels.h"
#include "tc_sm100.cuh"

namespace fcb {

using namespace tc;

constexpr int TC_M = 128;          // time rows per tile
constexpr int TC_KC = 32;          // channels per producer unit (half of a 128-byte fp16 swizzle row)
constexpr int TC_THREADS = 736;    // 16 producer warps (2 groups), copy warp, MMA warp, 4 accumulator warps, raw-tile TMA warp
constexpr int TC_RAW_MAX = 8;      // raw activation ring (TMA-staged units): at most 8 slots
constexpr int TC_PROD = 256;       // producer threads per group (one unit)
constexpr int TC_GROUP_MMAS = 48;  // target number of tcgen05.mma chained in TMEM before the fp32 fold

// ELU with the hardware exponential (ex2.approx): |error| <= ~2e-7 on the (0, 1] range of exp(x), the same order as
// one fp32 rounding of the reference's exp(x) - 1.  (The SIMT path keeps expf.)
__device__ __forceinline__ float elu_fast(float v) { return v > 0.f ? v : (__expf(v) - 1.0f); }
// the same on a value pre-multiplied by the operand scale s (a power of two): s*elu(v) from vs = s*v with k = log2(e)/s.
// Scaling by a power of two commutes with every rounding involved, so this equals s * elu_fast(v) bit for bit.
__device__ __forceinline__ float elu_scaled(float vs, float k, float s) { return vs > 0.f ? vs : fmaf(exp2f_approx(vs * k), s, -s); }

struct TcSmemLayout {
    int a_rows;        // rows per A slab (multiple of 8)
    int a_stage;       // bytes per A stage (hi + lo)
    int b_stage;       // bytes per B stage (hi + lo)
    int na, nb;        // ring depths
    int nraw, raw_slot, raw_in1, raw_cf;   // raw activation ring: slots, bytes per slot, offsets of in1 / coefficients in a slot
    int off_b, off_stg, off_raw, off_bar, total;
};

__host__ __device__ inline TcSmemLayout tc_layout(int K, int S, int n_tile, int na, int nb, int nraw = 0, int raw_pitch = 128,
                                                   int has1 = 0) {
    TcSmemLayout L;
    const int qmax = (K - 1) / S;
    L.a_rows = ((TC_M + qmax + 7) / 8) * 8;
    L.a_stage = 2 * L.a_rows * 128;
    L.b_stage = 2 * n_tile * 128;
    L.na = na; L.nb = nb;
    L.off_b = na * L.a_stage;
    L.off_stg = L.off_b + nb * L.b_stage;                  // epilogue staging: 4 warps x (32 rows x 128 B), swizzled
    // raw slot: [in0 rows][in1 rows][a0 | b0 | a1 | b1 coefficient slices of the unit's 32 channels (4 x 128 B)]
    L.nraw = nraw;
    L.raw_in1 = L.a_rows * raw_pitch;
    L.raw_cf = (1 + has1) * L.a_rows * raw_pitch;
    L.raw_slot = (L.raw_cf + 512 + 127) / 128 * 128;
    L.off_raw = L.off_stg + 4 * 4096;
    L.off_bar = L.off_raw + nraw * L.raw_slot;
    L.total = L.off_bar + 8 * (2 * na + 2 * nb + 16 + 2 * TC_RAW_MAX) + 96;
    return L;
}

// ring stages (64-channel chunk, phase) chained in one TMEM accumulation group
__host__ __device__ inline int tc_units_per_group(int K, int S, int group_mmas) {
    const int taps = (K + S - 1) / S;                  // max taps of a phase
    int g = group_mmas / (12 * taps);
    return g < 1 ? 1 : g;
}

// Launch-invariant quantities computed on the host and read from the kernel-parameter constant bank (instead of being
// derived -- and kept live in registers -- by every thread).
struct TcArgs {
    TcSmemLayout L;
    int na, nb, n_tiles, w_resident, nraw;
    int n_chunks, n_sc, split, n_units, upg, n_groups, n_tt, n_nt, units_per_tile, tq_rows, n_acc, raw_pitch;
};

struct TcTile { int b, nt, tt; };

__device__ __forceinline__ TcTile tc_tile(int id, int n_nt, int n_tt) {
    TcTile t;
    t.nt = id % n_nt;                  // n-tile fastest: concurrent CTAs share the activation rows in L2
    const int r = id / n_nt;
    t.tt = r % n_tt;
    t.b = r / n_tt;
    return t;
}

template <int N_TILE, bool FREQ>
__global__ void __launch_bounds__(TC_THREADS, 1) conv1d_tc_kernel(const __grid_constant__ ConvParams p, const __grid_constant__ TcArgs ka,
                                                                 const __grid_constant__ CUtensorMap tm0,
                                                                 const __grid_constant__ CUtensorMap tm1) {
    constexpr int BUF_COLS = N_TILE < 32 ? 32 : N_TILE;          // TMEM columns per accumulator region
    constexpr uint32_t TMEM_COLS = 512;                          // the whole TMEM: one CTA per SM
    constexpr int ACC_MAX = 8;                                   // accumulator ring: up to 8 tiles between MMA issue and epilogue
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int C_in = p.C_in, K = p.K, S = p.S;
    const bool has1 = p.in1.x != nullptr;
    const TcSmemLayout& L = ka.L;
#define na_stages ka.na
#define nb_stages ka.nb
#define n_tiles ka.n_tiles
#define w_resident ka.w_resident
#define nraw ka.nraw
#define raw_pitch ka.raw_pitch              /* bytes per row of a raw (TMA-staged) unit */
#define n_chunks ka.n_chunks                /* 32-channel chunks; C_in = 16: one half-empty chunk (zero channels, zero weights) */
#define n_sc ka.n_sc                        /* 64-channel stage chunks */
#define n_units ka.n_units                  /* ring stages per tile */
#define upg ka.upg
#define n_groups ka.n_groups
#define n_tt ka.n_tt
#define n_nt ka.n_nt
    const bool split = ka.split != 0;                     // both producer groups fill one stage (32 channels each)

    uint8_t* smA = smem_raw;
    uint8_t* smB = smem_raw + L.off_b;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + L.off_bar);
    uint64_t* a_full = bars;                       // [na]   128 producer arrivals (one group)
    uint64_t* a_empty = a_full + na_stages;        // [na]   tcgen05.commit
    uint64_t* b_full = a_empty + na_stages;        // [nb]   expect_tx
    uint64_t* b_empty = b_full + nb_stages;        // [nb]   tcgen05.commit
    uint64_t* acc_full = b_empty + nb_stages;      // [ACC_MAX] tcgen05.commit
    uint64_t* acc_empty = acc_full + ACC_MAX;      // [ACC_MAX] 128 accumulator-warp arrivals
    uint64_t* raw_full = acc_empty + ACC_MAX;      // [TC_RAW_MAX] expect_tx (TMA tile + coefficient slices)
    uint64_t* raw_empty = raw_full + TC_RAW_MAX;   // [TC_RAW_MAX] 256 arrivals of the consuming producer group
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(raw_empty + TC_RAW_MAX);
    uint8_t* smR = smem_raw + L.off_raw;
    // TMA-staged units (nraw > 0, 1-D layers): an INTERIOR tile needs only rows inside [0, rows covered by the tensor map) -- no
    // reflection, no zero padding -- so its units arrive as dense [a_rows][32 channel] boxes through the raw ring; the first / last
    // tiles of a clip keep the per-thread global loads (the index map lives there).  Units of a tile in ring order:
    // stage-major, half-minor; every role derives the slot from the same running count.
#define units_per_tile ka.units_per_tile
#define tq_rows ka.tq_rows                  /* rows per phase the tensor map exposes */
    auto tile_interior = [&](int t0) -> bool {
        if (nraw == 0) return false;
        // first / last input row that a VALID output row of the tile needs (a partial last tile only counts its real rows: the
        // rows a 1x1 layer does not have arrive zero-filled and feed discarded output rows only)
        const int t_last = (t0 + TC_M < p.T_out ? t0 + TC_M : p.T_out) - 1;
        const int lo = t0 * S - p.pad_l;
        const int hi = t_last * S - p.pad_l + (K - 1);
        return lo >= 0 && hi < tq_rows * S;
    };
    // accumulator ring depth.  The MMA -> commit -> epilogue -> release hand-off costs ~2000 cycles per tile pair (measured: the
    // pure barrier skeleton of the small-tile layers), so layers whose tile is one accumulation group keep up to 8 tiles in
    // flight; layers that fold groups (deep K) ping-pong between up to 3 accumulators next to the running totals.
#define n_acc ka.n_acc
    double* red = reinterpret_cast<double*>(tmem_ptr + 2);       // [4][2] statistics scratch

    if (tid == 0) {
        for (int i = 0; i < na_stages; ++i) { mbar_init(a_full + i, split ? 2 * TC_PROD : TC_PROD); mbar_init(a_empty + i, 1); }
        for (int i = 0; i < nb_stages; ++i) { mbar_init(b_full + i, 1); mbar_init(b_empty + i, 1); }
        for (int i = 0; i < ACC_MAX; ++i) { mbar_init(acc_full + i, 1); mbar_init(acc_empty + i, 128); }
        for (int i = 0; i < TC_RAW_MAX; ++i) { mbar_init(raw_full + i, 1); mbar_init(raw_empty + i, TC_PROD); }
        mbar_fence_init();
    }
    if (warp == 16) tmem_alloc(tmem_ptr, TMEM_COLS);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp < 16) {
        // =========================================================== producers: transformed A slabs
        const int grp = warp >> 3;
        const int ptid = tid & (TC_PROD - 1);
        const int jchunk = ptid & 7;                // 4 channels (16 bytes of fp32 in HBM, 8 bytes of fp16 in the slab)
        // rows of a warp: {b, b+1, b+4, b+5}: its four 64-byte half rows land on all 32 banks (2 wavefronts per 8-byte store)
        const int wq = (ptid >> 5), lq = (lane >> 3);
        const int rsub = ((wq >> 1) << 3) + ((wq & 1) << 1) + (lq & 1) + ((lq >> 1) << 2);      // 32 rows per pass
        const int gt_max = (p.T_out - 1) * S - p.pad_l + (K - 1);
        // this group's cursor over the CTA's global stage sequence (tile-major).  split: both groups fill every stage (group g
        // writes the 32-channel half g); otherwise (one 32-channel chunk) the groups take alternate stages and the ring slot
        // advances two at a time (na is even), so no division / modulo is needed in the loop
        const int step = split ? 1 : 2;
        const int half = split ? grp : 0;
        int tile = blockIdx.x, unit = split ? 0 : grp;
        int as = unit % na_stages;
        uint32_t aphase = 0;
        const float in_scale = p.tc_in_scale;
        int rawbase = 0;                            // raw-ring units of the interior tiles this CTA has passed
        while (unit >= n_units && tile < n_tiles) {
            if (tile_interior(tc_tile(tile, n_nt, n_tt).tt * TC_M)) rawbase += units_per_tile;
            unit -= n_units; tile += gridDim.x;
        }
        while (tile < n_tiles) {
            const TcTile tl = tc_tile(tile, n_nt, n_tt);
            const int t0 = tl.tt * TC_M;
            int b = tl.b, f_out = 0;
            if (FREQ) { b = tl.b / p.fq.F_out; f_out = tl.b - b * p.fq.F_out; }
            const int pitch = FREQ ? p.fq.cin : C_in;          // channels per stored input row
            const float* x0 = p.in0.x + (long long)b * p.in0.clip_stride + (long long)p.in0.row_off * pitch;
            const float* x1 = has1 ? p.in1.x + (long long)b * p.in1.clip_stride + (long long)p.in1.row_off * pitch : nullptr;
            const float* cf0 = p.in0.coef ? p.in0.coef + (long long)b * 2 * pitch : nullptr;
            const float* cf1 = (has1 && p.in1.coef) ? p.in1.coef + (long long)b * 2 * pitch : nullptr;
            const int cur_tile = tile;
            const bool interior = tile_interior(t0);
            for (; unit < n_units && tile == cur_tile; ) {
                const int sc = unit / S, ph = unit - sc * S;
                const int chunk = 2 * sc + half;               // 32-channel chunk of this group (may not exist: odd n_chunks)
                const uint32_t par = aphase ^ 1;
                uint8_t* hi = smA + as * L.a_stage;
                uint8_t* lo = hi + L.a_rows * 128;
                const uint32_t c16 = (uint32_t)(half * 4 + (jchunk >> 1)), sub8 = (uint32_t)((jchunk & 1) << 3);
                if (chunk >= n_chunks) {
                    mbar_wait_backoff(a_empty + as, par, 64);      // missing half of the last stage: never read by the MMAs
                } else if (interior) {
                    // ---- TMA-staged unit: the dense [a_rows][32 ch] boxes (+ the coefficient slices) wait in the raw ring; rows go
                    // shared -> registers -> shared one at a time (no long-latency loads to batch, few live registers)
                    const bool c_ok = chunk * TC_KC + jchunk * 4 < C_in;
                    const int idx = 2 * S * sc + ((2 * sc + 1 < n_chunks) ? 2 * ph + half : ph);
                    const int rc = rawbase + idx;
                    const int rslot = rc % nraw;
                    mbar_wait(raw_full + rslot, (uint32_t)((rc / nraw) & 1));
                    const uint8_t* rb = smR + rslot * L.raw_slot;
                    float4 a0 = make_float4(in_scale, in_scale, in_scale, in_scale), b0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, b1 = b0;
                    if (!c_ok) { a0 = b0; a1 = b0; }
                    else {
                        if (cf0) {
                            a0 = *reinterpret_cast<const float4*>(rb + L.raw_cf + jchunk * 16); b0 = *reinterpret_cast<const float4*>(rb + L.raw_cf + 128 + jchunk * 16);
                            a0.x *= in_scale; a0.y *= in_scale; a0.z *= in_scale; a0.w *= in_scale;
                            b0.x *= in_scale; b0.y *= in_scale; b0.z *= in_scale; b0.w *= in_scale;
                        }
                        if (cf1) {
                            a1 = *reinterpret_cast<const float4*>(rb + L.raw_cf + 256 + jchunk * 16); b1 = *reinterpret_cast<const float4*>(rb + L.raw_cf + 384 + jchunk * 16);
                            a1.x *= in_scale; a1.y *= in_scale; a1.z *= in_scale; a1.w *= in_scale;
                            b1.x *= in_scale; b1.y *= in_scale; b1.z *= in_scale; b1.w *= in_scale;
                        }
                    }
                    mbar_wait_backoff(a_empty + as, par, 64);
                    const uint8_t* rrow = rb + rsub * raw_pitch + jchunk * 16;
#pragma unroll
                    for (int i = 0; i < 5; ++i) {
                        const int u = rsub + 32 * i;
                        if (u < L.a_rows) {
                            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (c_ok) {
                                const float4 xv = *reinterpret_cast<const float4*>(rrow + i * 32 * raw_pitch);
                                v.x = fmaf(xv.x, a0.x, b0.x); v.y = fmaf(xv.y, a0.y, b0.y);
                                v.z = fmaf(xv.z, a0.z, b0.z); v.w = fmaf(xv.w, a0.w, b0.w);
                                if (has1) {
                                    const float4 yv = *reinterpret_cast<const float4*>(rrow + L.raw_in1 + i * 32 * raw_pitch);
                                    v.x = v.x + fmaf(yv.x, a1.x, b1.x); v.y = v.y + fmaf(yv.y, a1.y, b1.y);
                                    v.z = v.z + fmaf(yv.z, a1.z, b1.z); v.w = v.w + fmaf(yv.w, a1.w, b1.w);
                                }
                                if (p.elu) {
                                    v.x = elu_scaled(v.x, p.tc_elu_k, in_scale); v.y = elu_scaled(v.y, p.tc_elu_k, in_scale);
                                    v.z = elu_scaled(v.z, p.tc_elu_k, in_scale); v.w = elu_scaled(v.w, p.tc_elu_k, in_scale);
                                }
                            }
                            uint2 h, l;
                            split_f16x2(v.x, v.y, h.x, l.x);
                            split_f16x2(v.z, v.w, h.y, l.y);
                            const uint32_t o = (uint32_t)u * 128u + ((c16 ^ (uint32_t)(u & 7)) << 4) + sub8;
                            *reinterpret_cast<uint2*>(hi + o) = h;
                            *reinterpret_cast<uint2*>(lo + o) = l;
                        }
                    }
                    mbar_arrive(raw_empty + rslot);            // the raw rows have been consumed
                    fence_proxy_async_smem();
                } else {
                int c = chunk * TC_KC + jchunk * 4;
                bool c_ok = c < C_in;
                const float* xu0 = x0;
                const float* xu1 = x1;
                if (FREQ) {
                    // gathered channel -> (frequency tap, stored channel); the tap selects the input row of this thread
                    const int kf = c / pitch;
                    c -= kf * pitch;
                    int f_src = f_out * p.fq.SF + kf - p.fq.pad_f;
                    if (p.pad_zero) c_ok = c_ok && f_src >= 0 && f_src < p.fq.F_in;
                    else f_src = reflect_index(f_src, p.fq.F_in);
                    if (!c_ok) f_src = 0;
                    xu0 = x0 + (long long)(p.fq.f_off0 + f_src) * p.fq.T_raw0 * pitch;
                    if (has1) xu1 = x1 + (long long)(p.fq.f_off1 + f_src) * p.fq.T_raw1 * pitch;
                }
                // the operand scale (a power of two: exact) is folded into the deferred-GroupNorm affine
                float4 a0 = make_float4(in_scale, in_scale, in_scale, in_scale), b0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, b1 = b0;
                if (!c_ok) { a0 = b0; a1 = b0; }
                else if (cf0) {
                    a0 = __ldg(reinterpret_cast<const float4*>(cf0 + c)); b0 = __ldg(reinterpret_cast<const float4*>(cf0 + pitch + c));
                    a0.x *= in_scale; a0.y *= in_scale; a0.z *= in_scale; a0.w *= in_scale;
                    b0.x *= in_scale; b0.y *= in_scale; b0.z *= in_scale; b0.w *= in_scale;
                }
                if (c_ok && cf1) {
                    a1 = __ldg(reinterpret_cast<const float4*>(cf1 + c)); b1 = __ldg(reinterpret_cast<const float4*>(cf1 + pitch + c));
                    a1.x *= in_scale; a1.y *= in_scale; a1.z *= in_scale; a1.w *= in_scale;
                    b1.x *= in_scale; b1.y *= in_scale; b1.z *= in_scale; b1.w *= in_scale;
                }
                // all row loads of the unit are issued before the ring slot is waited for
                constexpr int NR = 5;                      // a_rows <= 160 = 5 passes of 32 rows
                float4 xa[NR], xb[NR];
                bool okr[NR];
#pragma unroll
                for (int i = 0; i < NR; ++i) {
                    const int u = rsub + 32 * i;
                    const int gt = (t0 + u) * S + ph - p.pad_l;
                    bool ok = c_ok && u < L.a_rows && gt <= gt_max;
                    int src = gt;
                    if (p.pad_zero) ok = ok && gt >= 0 && gt < p.T_in;
                    else { src = reflect_index(gt, p.T_ext); ok = ok && src < p.T_in && src >= 0; }
                    okr[i] = ok;
                    xa[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                    xb[i] = xa[i];
                    if (ok) {
                        const long long off = (long long)src * pitch + c;
                        xa[i] = __ldg(reinterpret_cast<const float4*>(xu0 + off));
                        if (has1) xb[i] = __ldg(reinterpret_cast<const float4*>(xu1 + off));
                    }
                }
                mbar_wait_backoff(a_empty + as, par, 64);
#pragma unroll
                for (int i = 0; i < NR; ++i) {
                    const int u = rsub + 32 * i;
                    if (u < L.a_rows) {
                        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (okr[i]) {
                            const float4 xv = xa[i];
                            v.x = fmaf(xv.x, a0.x, b0.x); v.y = fmaf(xv.y, a0.y, b0.y);
                            v.z = fmaf(xv.z, a0.z, b0.z); v.w = fmaf(xv.w, a0.w, b0.w);
                            if (has1) {
                                const float4 yv = xb[i];
                                v.x = v.x + fmaf(yv.x, a1.x, b1.x); v.y = v.y + fmaf(yv.y, a1.y, b1.y);
                                v.z = v.z + fmaf(yv.z, a1.z, b1.z); v.w = v.w + fmaf(yv.w, a1.w, b1.w);
                            }
                            if (p.elu) {
                                v.x = elu_scaled(v.x, p.tc_elu_k, in_scale); v.y = elu_scaled(v.y, p.tc_elu_k, in_scale);
                                v.z = elu_scaled(v.z, p.tc_elu_k, in_scale); v.w = elu_scaled(v.w, p.tc_elu_k, in_scale);
                            }
                        }
                        uint2 h, l;
                        split_f16x2(v.x, v.y, h.x, l.x);
                        split_f16x2(v.z, v.w, h.y, l.y);
                        const uint32_t o = (uint32_t)u * 128u + ((c16 ^ (uint32_t)(u & 7)) << 4) + sub8;
                        *reinterpret_cast<uint2*>(hi + o) = h;
                        *reinterpret_cast<uint2*>(lo + o) = l;
                    }
                }
                fence_proxy_async_smem();
                }
                mbar_arrive(a_full + as);
                as += step;
                if (as >= na_stages) { as -= na_stages; aphase ^= 1; }
                unit += step;
            }
            while (unit >= n_units && tile < n_tiles) {
                if (tile_interior(tc_tile(tile, n_nt, n_tt).tt * TC_M)) rawbase += units_per_tile;
                unit -= n_units; tile += gridDim.x;
            }
        }
    } else if (warp == 16) {
        // =========================================================== weight slabs via the bulk-copy engine
        if (lane == 0) {
            const uint32_t bytes = (uint32_t)L.b_stage;
            int bs = 0;
            uint32_t bphase = 0;
            bool first = true;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                if (w_resident && !first) break;                       // whole layer image already resident
                const TcTile tl = tc_tile(tile, n_nt, n_tt);
                const uint8_t* wbase = reinterpret_cast<const uint8_t*>(p.w_tc) + (long long)tl.nt * n_sc * K * bytes;
                int chunk = 0, ph = 0;                                 // chunk: 64-channel stage chunk
                for (int unit = 0; unit < n_units; ++unit) {
                    for (int k = ph; k < K; k += S) {
                        if (!w_resident) mbar_wait_backoff(b_empty + bs, bphase ^ 1, 64);
                        mbar_arrive_expect_tx(b_full + bs, bytes);
                        bulk_g2s(smB + bs * L.b_stage, wbase + ((long long)chunk * K + k) * bytes, bytes, b_full + bs);
                        if (++bs == nb_stages) { bs = 0; bphase ^= 1; }
                    }
                    if (++ph == S) { ph = 0; ++chunk; }
                }
                first = false;
            }
        }
    } else if (warp == 17) {
        // =========================================================== MMA issuer
        if (lane == 0) {
            const uint32_t idesc = make_idesc_f16(TC_M, N_TILE);
            const uint32_t a_base = smem_u32(smA), b_base = smem_u32(smB);
            int as = 0, bs = 0, buf = 0;
            uint32_t aphase = 0, bphase = 0, cphase = 0;
            bool first = true;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                int ph = 0;
                if (w_resident) bs = 0;
                for (int g = 0; g < n_groups; ++g) {
                    mbar_wait(acc_empty + buf, cphase ^ 1);
                    tc_fence_after_sync();
                    const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BUF_COLS);
                    uint32_t accum = 0;
                    const int u_end = min(n_units, (g + 1) * upg);
                    for (int unit = g * upg; unit < u_end; ++unit) {
                        mbar_wait(a_full + as, aphase);
                        tc_fence_after_sync();
                        const uint32_t a_hi0 = a_base + as * L.a_stage;
                        const uint32_t a_lo0 = a_hi0 + L.a_rows * 128;
                        // K steps of 16 channels: 4 for a full 64-channel stage, 2 when only its first half exists
                        const int ksteps = (2 * (unit / S) + 1 < n_chunks) ? 4 : 2;
                        int q = 0;
                        for (int k = ph; k < K; k += S, ++q) {
                            if (!w_resident || first) {
                                mbar_wait(b_full + bs, bphase);
                                tc_fence_after_sync();
                            }
                            const uint32_t b_hi0 = b_base + bs * L.b_stage;
                            const uint32_t b_lo0 = b_hi0 + N_TILE * 128;
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                if (ks < ksteps) {
                                    const uint64_t da_hi = make_desc_k_sw128(a_hi0 + q * 128 + ks * 32);
                                    const uint64_t da_lo = make_desc_k_sw128(a_lo0 + q * 128 + ks * 32);
                                    const uint64_t db_hi = make_desc_k_sw128(b_hi0 + ks * 32);
                                    const uint64_t db_lo = make_desc_k_sw128(b_lo0 + ks * 32);
                                    mma_f16_ss(d_tmem, da_lo, db_hi, idesc, accum);
                                    accum = 1;
                                    mma_f16_ss(d_tmem, da_hi, db_lo, idesc, 1);
                                    mma_f16_ss(d_tmem, da_hi, db_hi, idesc, 1);
                                }
                            }
                            if (!w_resident) mma_commit(b_empty + bs);
                            if (++bs == nb_stages) { bs = 0; bphase ^= 1; }
                        }
                        mma_commit(a_empty + as);
                        if (++as == na_stages) { as = 0; aphase ^= 1; }
                        if (++ph == S) ph = 0;
                    }
                    mma_commit(acc_full + buf);
                    if (++buf == n_acc) { buf = 0; cphase ^= 1; }
                }
                first = false;
            }
        }
    } else if (warp == 22) {
        // =========================================================== raw activation tiles via TMA (cp.async.bulk.tensor)
        if (lane == 0 && nraw > 0) {
            const uint32_t row_bytes = (uint32_t)(L.a_rows * raw_pitch);
            const uint32_t cbytes = (uint32_t)raw_pitch;
            const uint32_t n_cf = (p.in0.coef ? 2u : 0u) + ((has1 && p.in1.coef) ? 2u : 0u);
            const uint32_t unit_bytes = row_bytes * (has1 ? 2u : 1u) + n_cf * cbytes;
            int rc = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const TcTile tl = tc_tile(tile, n_nt, n_tt);
                const int t0 = tl.tt * TC_M;
                if (!tile_interior(t0)) continue;
                const int b = tl.b;
                const float* cf0 = p.in0.coef ? p.in0.coef + (long long)b * 2 * C_in : nullptr;
                const float* cf1 = (has1 && p.in1.coef) ? p.in1.coef + (long long)b * 2 * C_in : nullptr;
                for (int sc = 0; sc < n_sc; ++sc)
                    for (int ph = 0; ph < S; ++ph) {
                        // row (t0 + u) * S + ph - pad_l == (tq0 + u) * S + php
                        const int r = ph - p.pad_l;
                        const int fd = (r >= 0) ? r / S : -((-r + S - 1) / S);
                        const int tq0 = t0 + fd, php = r - fd * S;
                        for (int hh = 0; hh < 2; ++hh) {
                            const int chunk = 2 * sc + hh;
                            if (chunk >= n_chunks) break;
                            const int slot = rc % nraw;
                            mbar_wait(raw_empty + slot, (uint32_t)((rc / nraw) & 1) ^ 1);
                            uint8_t* dst = smR + slot * L.raw_slot;
                            mbar_arrive_expect_tx(raw_full + slot, unit_bytes);
                            const int c0 = chunk * TC_KC;      // first channel of the unit
                            tma_load_4d(dst, &tm0, c0, php, tq0, b, raw_full + slot);
                            if (has1) tma_load_4d(dst + L.raw_in1, &tm1, c0, php, tq0, b, raw_full + slot);
                            if (cf0) {
                                bulk_g2s(dst + L.raw_cf, cf0 + c0, cbytes, raw_full + slot);
                                bulk_g2s(dst + L.raw_cf + 128, cf0 + C_in + c0, cbytes, raw_full + slot);
                            }
                            if (cf1) {
                                bulk_g2s(dst + L.raw_cf + 256, cf1 + c0, cbytes, raw_full + slot);
                                bulk_g2s(dst + L.raw_cf + 384, cf1 + C_in + c0, cbytes, raw_full + slot);
                            }
                            ++rc;
                        }
                    }
            }
        }
    } else {
        // =========================================================== accumulator warps: fold groups, epilogue
        const int quad = warp & 3;                                   // a warp may only touch TMEM lanes 32*(warp%4)..+31
        const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
        const uint32_t tot_base = tmem_base + lane_base + (uint32_t)(n_acc * BUF_COLS);
        int buf = 0;
        uint32_t cphase = 0;
        // 2-D plain convs (no phase scatter, no padded columns) store [pseudo-clip][t][C_out] like a 1-D layer
        const bool plain_out = FREQ && p.fq.FR == 1 && p.fq.TR == 1 && p.fq.c_store == p.C_out;
        const float out_scale = p.tc_out_scale;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const TcTile tl = tc_tile(tile, n_nt, n_tt);
            const int t = tl.tt * TC_M + quad * 32 + lane;
            const bool row_ok = t < p.T_out;
            float* orow = p.out + (long long)tl.b * p.out_clip_stride + (long long)t * p.C_out + (long long)tl.nt * N_TILE;
            const float* bias = p.bias + tl.nt * N_TILE;
            long long frow = 0;                                       // FREQ: element row of (clip, f_out*FR, t*TR)
            if (FREQ) {
                const int fb = tl.b / p.fq.F_out, ff = tl.b - fb * p.fq.F_out;
                frow = ((long long)fb * p.fq.F_out * p.fq.FR + (long long)ff * p.fq.FR) * ((long long)p.T_out * p.fq.TR) + (long long)t * p.fq.TR;
            }
            float s = 0.f, ss = 0.f;
            for (int g = 0; g < n_groups; ++g) {
                const bool last = (g == n_groups - 1);
                mbar_wait_backoff(acc_full + buf, cphase, 128);
                tc_fence_after_sync();
#pragma unroll
                for (int c0 = 0; c0 < N_TILE; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld_32x32b_x32(tmem_base + lane_base + (uint32_t)(buf * BUF_COLS + c0), v);
                    if (g > 0) {
                        uint32_t tv[32];
                        tmem_ld_32x32b_x32(tot_base + (uint32_t)c0, tv);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(tv[j]) + __uint_as_float(v[j]));
                    } else {
                        tmem_ld_wait();
                    }
                    if (!last) {
                        tmem_st_32x32b_x32(tot_base + (uint32_t)c0, v);
                    } else if (!FREQ || plain_out) {
                        // bias + statistics in registers, then through a swizzled staging tile so that every global store
                        // instruction of the warp writes whole rows (4 rows x 128 B = 4 L1 wavefronts instead of 32)
                        uint8_t* stg = smem_raw + L.off_stg + quad * 4096;
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            if (c0 + j < N_TILE) {
                                float4 o;
                                o.x = fmaf(__uint_as_float(v[j + 0]), out_scale, __ldg(bias + c0 + j + 0));
                                o.y = fmaf(__uint_as_float(v[j + 1]), out_scale, __ldg(bias + c0 + j + 1));
                                o.z = fmaf(__uint_as_float(v[j + 2]), out_scale, __ldg(bias + c0 + j + 2));
                                o.w = fmaf(__uint_as_float(v[j + 3]), out_scale, __ldg(bias + c0 + j + 3));
                                if (row_ok) {
                                    s += (o.x + o.y) + (o.z + o.w);
                                    ss = fmaf(o.x, o.x, ss); ss = fmaf(o.y, o.y, ss); ss = fmaf(o.z, o.z, ss); ss = fmaf(o.w, o.w, ss);
                                }
                                *reinterpret_cast<float4*>(stg + lane * 128 + ((((j >> 2) ^ (lane & 7))) << 4)) = o;
                            }
                        }
                        __syncwarp();
                        const int cc = lane & 7;
                        if (c0 + cc * 4 < N_TILE) {
                            float* obase = p.out + (long long)tl.b * p.out_clip_stride + (long long)tl.nt * N_TILE + c0 + cc * 4;
                            const int trow0 = tl.tt * TC_M + quad * 32;
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const int rr = i * 4 + (lane >> 3);
                                if (trow0 + rr < p.T_out)
                                    *reinterpret_cast<float4*>(obase + (long long)(trow0 + rr) * p.C_out) =
                                        *reinterpret_cast<const float4*>(stg + rr * 128 + ((cc ^ (rr & 7)) << 4));
                            }
                        }
                        __syncwarp();
                    } else if (row_ok) {
                        int ph = 0, cch = 0;                          // FREQ: phase and channel of output column c0 + j
                        {
                            const int co = tl.nt * N_TILE + c0;
                            ph = co / p.fq.Cc;
                            cch = co - ph * p.fq.Cc;
                        }
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            if (c0 + j < N_TILE) {
                                float4 o;
                                // exact power-of-two rescale + bias in one rounding (== fl(acc / scale + bias))
                                o.x = fmaf(__uint_as_float(v[j + 0]), out_scale, __ldg(bias + c0 + j + 0));
                                o.y = fmaf(__uint_as_float(v[j + 1]), out_scale, __ldg(bias + c0 + j + 1));
                                o.z = fmaf(__uint_as_float(v[j + 2]), out_scale, __ldg(bias + c0 + j + 2));
                                o.w = fmaf(__uint_as_float(v[j + 3]), out_scale, __ldg(bias + c0 + j + 3));
                                s += (o.x + o.y) + (o.z + o.w);
                                ss = fmaf(o.x, o.x, ss); ss = fmaf(o.y, o.y, ss); ss = fmaf(o.z, o.z, ss); ss = fmaf(o.w, o.w, ss);
                                // phase (pf, pt) of a transposed conv lands on row f_out*FR + pf, column t*TR + pt
                                const int pf = ph / p.fq.TR, pt = ph - pf * p.fq.TR;
                                float* dst = p.out + (frow + (long long)pf * p.T_out * p.fq.TR + pt) * p.fq.c_store + cch;
                                if ((p.fq.c_store & 3) == 0) {
                                    if (cch < p.fq.c_store) *reinterpret_cast<float4*>(dst) = o;   // (padded columns: no store)
                                } else {                          // padded n-tile: only the real channels exist in HBM
                                    if (cch + 0 < p.fq.c_store) dst[0] = o.x;
                                    if (cch + 1 < p.fq.c_store) dst[1] = o.y;
                                    if (cch + 2 < p.fq.c_store) dst[2] = o.z;
                                    if (cch + 3 < p.fq.c_store) dst[3] = o.w;
                                }
                                cch += 4;
                                if (cch >= p.fq.Cc) { cch = 0; ++ph; }
                            }
                        }
                    }
                }
                if (!last) tmem_st_wait();
                tc_fence_before_sync();
                mbar_arrive(acc_empty + buf);
                if (++buf == n_acc) { buf = 0; cphase ^= 1; }
            }
            if (p.partials) {
                double ds = (double)s, dss = (double)ss;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    ds += __shfl_xor_sync(0xffffffffu, ds, o);
                    dss += __shfl_xor_sync(0xffffffffu, dss, o);
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");      // previous tile's reader is done with `red`
                if (lane == 0) { red[quad * 2] = ds; red[quad * 2 + 1] = dss; }
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (quad == 0 && lane == 0) {
                    const int nparts = n_nt * n_tt;
                    double* dst = p.partials + ((long long)tl.b * nparts + tl.nt * n_tt + tl.tt) * 2;
                    dst[0] = (red[0] + red[2]) + (red[4] + red[6]);
                    dst[1] = (red[1] + red[3]) + (red[5] + red[7]);
                }
            }
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 16) {
        tc_fence_after_sync();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
#undef na_stages
#undef nb_stages
#undef n_tiles
#undef w_resident
#undef nraw
#undef raw_pitch
#undef n_chunks
#undef n_sc
#undef n_units
#undef upg
#undef n_groups
#undef n_tt
#undef n_nt
#undef units_per_tile
#undef tq_rows
#undef n_acc
}

// ------------------------------------------------------------------------------------------ host side
bool conv_tc_supported(int C_in, int C_out_eff, int K, int S, int D) {
    return D == 1 && (C_in % TC_KC == 0 || C_in == 16) && C_out_eff % 16 == 0 && K >= 1 && S >= 1 && ((K - 1) / S) <= 16;
}

// 2-D mode: cin stored channels per input element, C_out_eff output columns of the (possibly n-tile padded) weight image
bool conv_tc_supported_2d(int cin, int C_out_eff, int KT, int ST) {
    const bool cin_ok = cin % 4 == 0 && (cin % TC_KC == 0 || TC_KC % cin == 0);   // a thread's 4 channels share one tap
    return cin_ok && C_out_eff % 16 == 0 && KT >= 1 && ST >= 1 && ((KT - 1) / ST) <= 16;
}

int conv_tc_n_tile(int C_out_eff) {
    if (C_out_eff >= 128 && C_out_eff % 128 == 0) return 128;
    if (C_out_eff % 64 == 0) return 64;
    if (C_out_eff % 32 == 0) return 32;
    return 16;
}

int conv_tc_num_parts(int T_out, int C_out_eff) {
    return ((T_out + TC_M - 1) / TC_M) * (C_out_eff / conv_tc_n_tile(C_out_eff));
}

static int g_num_sms = 0;

struct TcPlan { int resident, na, nb, nraw; TcSmemLayout L; bool ok; };

// shared-memory plan: weights resident (small layers: the whole image of the single n-tile) or streamed through a ring as
// deep as fits; A ring `na_first` stages (4, else 2) -- with a raw TMA ring the A ring only decouples producers from the MMA
// issue, so 2 stages suffice and the rest of the shared memory buys prefetch depth (nraw units in flight).
static TcPlan tc_plan(const ConvParams& p, int na_first, bool want_raw) {
    const int limit = 225 * 1024;
    const int n_slabs = ((p.C_in + 2 * TC_KC - 1) / (2 * TC_KC)) * p.K;   // (64-channel stage chunk, tap) weight slabs per n-tile
    const int has1 = p.in1.x ? 1 : 0;
    const int raw_pitch = (p.C_in < TC_KC ? p.C_in : TC_KC) * 4;           // raw ring: 1-D layers only
    TcPlan pl{};
    pl.ok = false;
    int na = na_first, nb = 4;
    TcSmemLayout L = tc_layout(p.K, p.S, p.n_tile, na, n_slabs);
    const int min_raw = want_raw ? 2 : 0;
    auto fits = [&](const TcSmemLayout& l) { return l.total + min_raw * tc_layout(p.K, p.S, p.n_tile, 2, 2, 1, raw_pitch, has1).raw_slot <= limit; };
    if (n_slabs <= 64 && p.C_out == p.n_tile && fits(L)) { pl.resident = 1; nb = n_slabs; }   // one n-tile only
    else {
        L = tc_layout(p.K, p.S, p.n_tile, na, nb);
        if (!fits(L)) { nb = 3; L = tc_layout(p.K, p.S, p.n_tile, na, nb); }
        if (!fits(L)) { na = 2; nb = 4; L = tc_layout(p.K, p.S, p.n_tile, na, nb); }
        if (!fits(L)) { nb = 3; L = tc_layout(p.K, p.S, p.n_tile, na, nb); }
        if (!fits(L)) { nb = 2; L = tc_layout(p.K, p.S, p.n_tile, na, nb); }
        if (!fits(L)) return pl;
        // small n-tiles: a weight slab is only n_tile*256 bytes, so the ring is deepened until shared memory is full
        if (!want_raw)
            while (nb < 24 && nb < n_slabs && tc_layout(p.K, p.S, p.n_tile, na, nb + 1).total <= limit)
                L = tc_layout(p.K, p.S, p.n_tile, na, ++nb);
    }
    int nraw = 0;
    if (want_raw) {
        nraw = 2;
        while (nraw < TC_RAW_MAX && tc_layout(p.K, p.S, p.n_tile, na, nb, nraw + 1, raw_pitch, has1).total <= limit) ++nraw;
    }
    pl.L = tc_layout(p.K, p.S, p.n_tile, na, nb, nraw, raw_pitch, has1);
    pl.na = na; pl.nb = nb; pl.nraw = nraw;
    pl.ok = pl.L.total <= limit;
    return pl;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode_tiled = nullptr;
static int g_tma_state = 0;      // 0: not probed, 1: available, -1: unavailable

// 4-D view of a channels-last activation [B][T][C] that makes every stride phase a dimension: (channel, phase, row / S, clip).
// A unit of a tile = box {32 channels, 1 phase, a_rows rows, 1 clip}; rows beyond T / S (and before 0) are zero-filled.
static bool make_act_map(CUtensorMap* tm, const InView& v, int C, int S, int T_in, int B, int a_rows) {
    const float* base = v.x + (long long)v.row_off * C;
    const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)S, (cuuint64_t)(T_in / S), (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)C * 4, (cuuint64_t)S * C * 4, (cuuint64_t)v.clip_stride * 4};
    const cuuint32_t box[4] = {(cuuint32_t)(C < TC_KC ? C : TC_KC), 1, (cuuint32_t)a_rows, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    if (((uintptr_t)base & 15) != 0 || (strides[0] & 15) || (strides[2] & 15) || dims[2] == 0) return false;
    return g_encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int N_TILE, bool FREQ>
static cudaError_t launch_tc_n(const ConvParams& p, cudaStream_t st, const TcPlan& pl, int n_tiles, const CUtensorMap& tm0,
                               const CUtensorMap& tm1) {
    auto kern = conv1d_tc_kernel<N_TILE, FREQ>;
    {
        cudaError_t e = ensure_dynamic_smem((const void*)kern, 225 * 1024);
        if (e != cudaSuccess) return e;
    }
    const int grid = n_tiles < g_num_sms ? n_tiles : g_num_sms;
    TcArgs ka{};
    ka.L = pl.L; ka.na = pl.na; ka.nb = pl.nb; ka.n_tiles = n_tiles; ka.w_resident = pl.resident; ka.nraw = pl.nraw;
    ka.n_chunks = (p.C_in + TC_KC - 1) / TC_KC;
    ka.n_sc = (ka.n_chunks + 1) >> 1;
    ka.split = ka.n_chunks > 1;
    ka.n_units = ka.n_sc * p.S;
    ka.upg = tc_units_per_group(p.K, p.S, TC_GROUP_MMAS);
    ka.n_groups = (ka.n_units + ka.upg - 1) / ka.upg;
    ka.n_tt = (p.T_out + TC_M - 1) / TC_M;
    ka.n_nt = p.C_out / N_TILE;
    ka.units_per_tile = ka.n_chunks * p.S;
    ka.tq_rows = p.T_in / p.S;
    ka.raw_pitch = (p.C_in < TC_KC ? p.C_in : TC_KC) * 4;
    // accumulator ring depth: layers whose tile is one accumulation group keep up to 8 tiles in flight between MMA issue and
    // epilogue; layers that fold groups (deep K) ping-pong between up to 3 accumulators next to the running totals
    constexpr int BUF_COLS = N_TILE < 32 ? 32 : N_TILE;
    const int acc_fit = 512 / BUF_COLS;
    ka.n_acc = ka.n_groups == 1 ? (acc_fit < 8 ? acc_fit : 8) : (acc_fit - 1 < 3 ? acc_fit - 1 : 3);
    kern<<<grid, TC_THREADS, pl.L.total, st>>>(p, ka, tm0, tm1);
    return cudaGetLastError();
}

template <int N_TILE>
static cudaError_t launch_tc_modes(const ConvParams& p, cudaStream_t st, const TcPlan& pl, int n_tiles, bool freq,
                                   const CUtensorMap& tm0, const CUtensorMap& tm1) {
    return freq ? launch_tc_n<N_TILE, true>(p, st, pl, n_tiles, tm0, tm1) : launch_tc_n<N_TILE, false>(p, st, pl, n_tiles, tm0, tm1);
}

cudaError_t launch_conv_tc(const ConvParams& p_in, int B, cudaStream_t st, int* nparts) {
    ConvParams p = p_in;
    if (g_num_sms == 0) {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        e = cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return e;
        // TMA staging of the activation tiles: cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda)
        g_tma_state = -1;
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && fn &&
            qres == cudaDriverEntryPointSuccess) {
            g_encode_tiled = (EncodeTiledFn)fn;
            g_tma_state = 1;
        }
    }
    if (!(p.tc_in_scale > 0.f)) p.tc_in_scale = 16.f;           // post-GroupNorm activations are O(1): 16 x keeps |x| < 4094 finite
    if (!(p.tc_w_scale > 0.f)) p.tc_w_scale = 1.f;
    p.tc_out_scale = 1.0f / (p.tc_in_scale * p.tc_w_scale);     // powers of two: exact
    p.tc_elu_k = 1.4426950408889634f / p.tc_in_scale;
    const int n_tt = (p.T_out + TC_M - 1) / TC_M, n_nt = p.C_out / p.n_tile;
    *nparts = n_tt * n_nt;
    const int n_tiles = n_tt * n_nt * B;
    const bool freq = p.fq.KF > 0;          // B counts pseudo-clips (clips x output frequency rows) in the 2-D mode
    // raw TMA ring: 1-D layers with interior tiles (n_tt >= 3), channel counts the box covers, 16-byte aligned views
    CUtensorMap tm0{}, tm1{};
    // (interior tiles exist when the clip has at least 3 tiles, or for 1x1 layers -- no halo -- always)
    // 2-D layers keep the per-thread gather: the K_F-fold re-read of every input row makes the unit stream L2-bound either way,
    // and staging it through the raw ring measured slower at config 4 (r2g: conv stack 37.3 vs 33.6 ms)
    bool want_raw = g_tma_state == 1 && !freq && (n_tt >= 3 || (p.K == 1 && p.S == 1 && p.pad_l == 0)) && p.T_in / p.S >= 1 &&
                    (p.C_in % TC_KC == 0 || p.C_in == 16);
    TcPlan pl{};
    if (want_raw) {
        pl = tc_plan(p, 2, true);
        want_raw = pl.ok && pl.nraw >= 2 && make_act_map(&tm0, p.in0, p.C_in, p.S, p.T_in, B, pl.L.a_rows) &&
                   (!p.in1.x || make_act_map(&tm1, p.in1, p.C_in, p.S, p.T_in, B, pl.L.a_rows));
    }
    if (!want_raw) {
        pl = tc_plan(p, 4, false);
        if (!pl.ok) return cudaErrorInvalidConfiguration;
    }
    switch (p.n_tile) {
        case 16: return launch_tc_modes<16>(p, st, pl, n_tiles, freq, tm0, tm1);
        case 32: return launch_tc_modes<32>(p, st, pl, n_tiles, freq, tm0, tm1);
        case 64: return launch_tc_modes<64>(p, st, pl, n_tiles, freq, tm0, tm1);
        case 128: return launch_tc_modes<128>(p, st, pl, n_tiles, freq, tm0, tm1);
        default: return cudaErrorInvalidConfiguration;
    }
}

}  // namespace fcb
