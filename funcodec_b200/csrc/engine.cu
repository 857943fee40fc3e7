// Host-side engine + C ABI (include/funcodec_b200.h): weight repacking, the layer walk of the SEANet
// encoder / decoder, the RVQ call and stream-ordered workspace management.
//
// Layer walk follows SEANetEncoder.__init__ (funcodec/models/encoder/seanet_encoder.py:108-162),
// SEANetDecoder.__init__ (funcodec/models/decoder/seanet_decoder.py:107-172) and Encodec._encode_frame /
// _decode_frame (funcodec/models/codec_basic.py:361-408).  Activations are raw channels-last tensors with
// deferred GroupNorm (common.cuh); temporaries come from the CUDA stream-ordered pool (cudaMallocAsync), so
// a whole call enqueues without host synchronisation and memory is recycled layer by layer.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/funcodec_b200.h"
#include "common.cuh"
#include "kernels.h"

using namespace fcb;

namespace {

struct HostTensor {
    std::vector<int64_t> shape;
    std::vector<float> data;
};

struct ConvW {           // one SConv1d / SConvTranspose1d, packed for conv1d_cl_kernel
    int cin = 0, cout = 0, k = 0, s = 1, d = 1;
    bool transposed = false;
    float* w = nullptr;      // [K_eff][cin][cout_eff]
    float* bias = nullptr;   // [cout_eff]
    float* gamma = nullptr;  // [cout]
    float* beta = nullptr;   // [cout]
    float* w_tc = nullptr;   // tensor-core image: [n_tile idx][64-ch chunk][tap][hi|lo][n_tile rows x 128 B swizzled fp16]
    float tc_scale = 1.f;    // power-of-two scale baked into w_tc (build_tc_image_f16)
    int n_tile = 0;          // 0: no tensor-core image (layer runs on the SIMT kernel)
};

struct LstmW {
    int H = 0, layers = 0;
    std::vector<ConvW> ih;                // input projections as 1x1 convs: [1][H][4H] + bias (b_ih + b_hh)
    std::vector<float*> whh;              // packed [H][4H]
    std::vector<float> whh_scale;         // power-of-two fp16 operand scale per layer (max|w| * scale in [2^13, 2^14))
};

struct ResBlockW { ConvW c1, c2, sc; };

// A raw activation plus its deferred GroupNorm.
struct Act {
    float* p = nullptr;
    int T = 0, C = 0;
    long long clip_stride = 0;
    int row_off = 0;
    float* stats = nullptr;          // [B][2] or nullptr (plain tensor)
    float* coef = nullptr;           // [B][2][C] per-channel affine of the deferred GroupNorm (with stats)
    const float* gamma = nullptr;
    const float* beta = nullptr;
    bool owned = false;              // p (and stats) were allocated from the pool by the engine
    long long ch_stride = 0;         // 0: channels-last; else channel-planar [B][C][T] (the stereo waveform), this channel stride
};

}  // namespace

struct fcb_handle {
    fcb_config cfg{};
    int device = 0;
    bool finalized = false;
    std::map<std::string, HostTensor> host;
    std::string err;
    int64_t launches = 0;

    ConvW enc_conv0, enc_final, dec_conv0, dec_final;
    std::vector<ResBlockW> enc_rb, dec_rb;
    std::vector<ConvW> enc_down, dec_up;
    LstmW enc_lstm, dec_lstm;
    float* embed = nullptr;   // [n_q][K][D]
    float* cnorm = nullptr;   // [n_q][K]
    float* embed_tc = nullptr; // tensor-core image of the codebooks (rvq_tc.cu)
    int* err_flag = nullptr;
    unsigned* lstm_barrier = nullptr;
    int rvq_sliced = 1;          // "rvq_sliced" option / FCB_RVQ_SLICED: the column-sliced fp32 RVQ kernel (rvq_simt.cu) for D > 260 (the
                                 // SoundStream YAMLs' D = 512; r2o found that such a D never fit the whole-chunk kernel).  Validated on
                                 // hardware in r2q (profiles/soundstream_fullwidth_r2q.txt: codes exact on 4 x 300 frames x 32 stages);
                                 // 0 makes fcb_finalize refuse such a D instead
    unsigned long long* lstm_trace = nullptr;   // PROFILING ONLY (env FCB_LSTM_TRACE): managed buffer, dumped by fcb_destroy
    bool use_tc = true;      // tensor-core conv path (FCB_DISABLE_TC=1 or fcb_set_option disables it)
    int use_tc2d = 7;        // FreqCodec 2-D layers on the tensor-core path, bit mask of Conv2W::tc_class ("use_tc2d" option)
    int stft_tc = 1;             // STFT / iSTFT as tensor-core GEMMs ("stft_tc" option; 0: the direct-DFT kernels)
    ConvW stft_w, istft_w;       // their basis matrices as conv_tc weight images (finalize_freq)
    bool stft_packed = false;
    int stft_ld = 0, istft_ld = 0;   // padded column counts: STFT output (2*n_bins -> x128), iSTFT input (2*n_bins -> x32)
    int conv2d_small_cout = 1;   // halo-tile SIMT kernel for the C_out <= 4 2-D conv ("conv2d_small_cout" option; 0: padded n-tile)
    std::vector<void*> dev_allocs;
    std::map<std::string, const ConvW*> by_name;   // reference module prefix -> packed layer (debug hook)

    // FreqCodec (arch 1) layers
    struct Conv2W {
        int cin = 0, cout = 0, kf = 0, kt = 0, sf = 1, st = 1;
        int kf_eff = 0, kt_eff = 0;   // taps of the conv actually executed (2 x 2 for a transposed conv)
        bool transposed = false;
        float* w = nullptr; float* bias = nullptr; float* gamma = nullptr; float* beta = nullptr;
        // tensor-core image (conv_tc.cu 2-D mode) of [kt][kf*cin][cout_tc]; cout_tc = C_out_eff rounded up to 16
        float* w_tc = nullptr; float* bias_tc = nullptr;
        float tc_scale = 1.f;
        int n_tile = 0, cout_tc = 0;
        int tc_class = 0;    // 1: cin % 32 == 0; 2: cin < 32 (several frequency taps per chunk); 4: padded C_out
        int out_pad[2][2] = {{0, 0}, {0, 0}};   // transposed conv out_padding {{f_l, f_r}, {t_l, t_r}} (conv.py:410-445)
    };
    struct ResBlock2W { Conv2W c1, c2, sc; };
    Conv2W f_enc_conv0, f_dec_final;
    std::vector<ResBlock2W> f_enc_rb, f_dec_rb;
    std::vector<Conv2W> f_enc_down, f_dec_up;
    std::map<std::string, const Conv2W*> by_name2; // same for the 2-D layers (fcb_debug_conv2d)

    bool profiling = false;
    cudaEvent_t ev[FCB_NUM_PHASES + 1][2]{};
    bool ev_used[FCB_NUM_PHASES]{};
    bool ev_created = false;

    int tprod() const { int h = 1; for (int i = 0; i < cfg.n_ratios; ++i) h *= cfg.ratios[i]; return h; }
    // samples per codec frame: prod(ratios), times the STFT hop for the FreqCodec variant
    int hop() const { return cfg.arch == 1 ? tprod() * cfg.stft_hop : tprod(); }
    int top_channels() const { return cfg.n_filters << cfg.n_ratios; }
    int channels() const { return cfg.channels == 2 ? 2 : 1; }   // audio channels (fcb_config.channels 0 / 1: mono)
};

namespace {

#define FCB_CK(call)                                                                              \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess) {                                                                 \
            char buf__[512];                                                                      \
            snprintf(buf__, sizeof buf__, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            h->err = buf__;                                                                       \
            return FCB_E_CUDA;                                                                    \
        }                                                                                         \
    } while (0)

#define FCB_TRY(expr)                  \
    do {                               \
        int rc__ = (expr);             \
        if (rc__ != FCB_OK) return rc__; \
    } while (0)

int fail(fcb_handle* h, int code, const std::string& msg) { h->err = msg; return code; }

// ------------------------------------------------------------------------------------------- weights
const HostTensor* find(fcb_handle* h, const std::string& name) {
    auto it = h->host.find(name);
    return it == h->host.end() ? nullptr : &it->second;
}

int upload(fcb_handle* h, const std::vector<float>& v, float** out) {
    float* d = nullptr;
    FCB_CK(cudaMalloc(&d, v.size() * sizeof(float)));
    h->dev_allocs.push_back(d);
    FCB_CK(cudaMemcpy(d, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
    *out = d;
    return FCB_OK;
}

int need(fcb_handle* h, const std::string& name, std::vector<int64_t> shape, const HostTensor** out) {
    const HostTensor* t = find(h, name);
    if (!t) return fail(h, FCB_E_MISSING, "missing tensor: " + name);
    if (t->shape != shape) return fail(h, FCB_E_INVALID, "shape mismatch for " + name);
    *out = t;
    return FCB_OK;
}

// fp32 -> fp16 bits, round-to-nearest-even, saturating to +-65504 (the device side uses cvt.rn.satfinite.f16x2.f32)
uint16_t f32_to_f16_bits(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    const uint32_t sign = (u >> 16) & 0x8000u;
    u &= 0x7FFFFFFFu;
    if (u >= 0x477FF000u) return (uint16_t)(sign | 0x7BFFu);            // >= 65520 (rounds past the largest finite) or inf / nan
    if (u < 0x38800000u) {                                               // < 2^-14: subnormal result, multiples of 2^-24
        float ax;
        memcpy(&ax, &u, 4);
        const float r = ax * 16777216.0f;                                // exact (power of two); |r| < 1024
        const float rr = nearbyintf(r);                                  // default rounding mode: nearest even
        return (uint16_t)(sign | (uint32_t)rr);
    }
    const uint32_t mant = u & 0x7FFFFFu, exp = (u >> 23) - 112u;         // rebias 127 -> 15
    uint32_t h = (exp << 10) | (mant >> 13);
    const uint32_t rem = mant & 0x1FFFu;
    if (rem > 0x1000u || (rem == 0x1000u && (h & 1u))) ++h;              // carries into the exponent correctly
    return (uint16_t)(sign | h);
}

float f16_bits_to_f32(uint16_t hb) {
    const uint32_t sign = (uint32_t)(hb & 0x8000u) << 16, e = (hb >> 10) & 0x1Fu, m = hb & 0x3FFu;
    float out;
    if (e == 0) {
        out = (float)m * (1.0f / 16777216.0f);
    } else {
        const uint32_t u = ((e + 112u) << 23) | (m << 13);
        memcpy(&out, &u, 4);
    }
    uint32_t u;
    memcpy(&u, &out, 4);
    u |= sign;
    memcpy(&out, &u, 4);
    return out;
}

// Tensor-core weight image (conv_tc.cu): for every (n-tile, 64-channel chunk, tap) one hi slab and one lo slab of
// [n_tile rows (output channels) x 64 fp16] in the canonical K-major SWIZZLE_128B layout, so that a single 1-D bulk copy
// drops it into shared memory ready for tcgen05.mma kind::f16.  The weights are multiplied by *scale_out = 2^e chosen so that
// max|w| lands in [2^13, 2^14) (well inside fp16, and the lo terms of all but negligible weights stay normal numbers);
// hi = fp16(w * scale), lo = fp16(w * scale - hi).  The image is returned as packed 32-bit words (two fp16 each).
void build_tc_image_f16(const std::vector<float>& wp /*[K][cin][cout_eff]*/, int K, int cin, int cout_eff, int n_tile,
                        std::vector<float>* img_out, float* scale_out) {
    float mx = 0.f;
    for (float v : wp) { const float a = fabsf(v); if (a > mx && a < INFINITY) mx = a; }
    float scale = 1.f;
    if (mx > 0.f) {
        int e = 0;
        frexpf(mx, &e);                       // mx = m * 2^e, m in [0.5, 1)
        int sh = 14 - e;                      // mx * 2^sh in [2^13, 2^14)
        if (sh > 40) sh = 40;
        if (sh < -40) sh = -40;
        scale = ldexpf(1.f, sh);
    }
    *scale_out = scale;
    const int n_chunks = (cin + 63) / 64, n_nt = cout_eff / n_tile;   // a partial last chunk is zero-padded
    const size_t slab = (size_t)n_tile * 32;                 // 32-bit words per hi (or lo) slab: n_tile rows x 128 bytes
    std::vector<float>& img = *img_out;
    img.assign((size_t)n_nt * n_chunks * K * 2 * slab, 0.f);
    for (int nt = 0; nt < n_nt; ++nt)
        for (int c = 0; c < n_chunks; ++c)
            for (int k = 0; k < K; ++k) {
                uint16_t* hi = reinterpret_cast<uint16_t*>(img.data() + (((size_t)nt * n_chunks + c) * K + k) * 2 * slab);
                uint16_t* lo = hi + 2 * slab;
                for (int n = 0; n < n_tile; ++n)
                    for (int col = 0; col < 64; ++col) {
                        const float x = (c * 64 + col < cin) ? wp[((size_t)k * cin + c * 64 + col) * cout_eff + nt * n_tile + n] * scale : 0.f;
                        const uint16_t xh = f32_to_f16_bits(x);
                        const uint16_t xl = f32_to_f16_bits(x - f16_bits_to_f32(xh));
                        const size_t off = (size_t)n * 64 + ((((col >> 3) ^ (n & 7)) << 3) | (col & 7));   // 16-byte chunk ^ (row & 7)
                        hi[off] = xh;
                        lo[off] = xl;
                    }
            }
}

// tf32 variant (rvq_tc.cu codebook slabs): for every (n-tile, 32-channel chunk, tap) one hi slab and one lo
// slab of [n_tile rows (output channels) x 32 tf32] in the canonical K-major SWIZZLE_128B layout.  hi/lo = 3xTF32 split.
void build_tc_image_tf32(const std::vector<float>& wp /*[K][cin][cout_eff]*/, int K, int cin, int cout_eff, int n_tile,
                          std::vector<float>* img_out) {
    const int n_chunks = (cin + 31) / 32, n_nt = cout_eff / n_tile;   // a partial last chunk is zero-padded
    const size_t slab = (size_t)n_tile * 32;                 // floats per hi (or lo) slab
    std::vector<float>& img = *img_out;
    img.assign((size_t)n_nt * n_chunks * K * 2 * slab, 0.f);
    for (int nt = 0; nt < n_nt; ++nt)
        for (int c = 0; c < n_chunks; ++c)
            for (int k = 0; k < K; ++k) {
                float* hi = img.data() + (((size_t)nt * n_chunks + c) * K + k) * 2 * slab;
                float* lo = hi + slab;
                for (int n = 0; n < n_tile; ++n)
                    for (int col = 0; col < 32; ++col) {
                        const float x = (c * 32 + col < cin) ? wp[((size_t)k * cin + c * 32 + col) * cout_eff + nt * n_tile + n] : 0.f;
                        uint32_t u;
                        memcpy(&u, &x, 4);
                        u = (u + 0x1000u) & 0xFFFFE000u;
                        float xh;
                        memcpy(&xh, &u, 4);
                        const size_t off = (size_t)n * 32 + ((((col >> 2) ^ (n & 7)) << 2) | (col & 3));
                        hi[off] = xh;
                        lo[off] = x - xh;
                    }
            }
}

int pack_tc(fcb_handle* h, const std::vector<float>& wp /*[K][cin][cout_eff]*/, int K, int cin, int cout_eff, ConvW* o) {
    o->n_tile = 0;
    if (!h->use_tc || !conv_tc_supported(cin, cout_eff, K, 1, o->d)) return FCB_OK;   // dilated convs run on the SIMT kernel
    const int n_tile = conv_tc_n_tile(cout_eff);
    std::vector<float> img;
    build_tc_image_f16(wp, K, cin, cout_eff, n_tile, &img, &o->tc_scale);
    FCB_TRY(upload(h, img, &o->w_tc));
    o->n_tile = n_tile;
    return FCB_OK;
}

// Effective weight of a NormConv1d / NormConvTranspose1d (conv.py:25-35,148-202).  `norm: time_group_norm` stores the plain
// `.weight`; `norm: weight_norm` stores torch.nn.utils.weight_norm's `.weight_g` [d0,1,1] and `.weight_v` (dim 0: output
// channels of a Conv1d, INPUT channels of a ConvTranspose1d) and the module computes w = v * (g / ||v||_2 over the other dims)
// (ATen _weight_norm); a checkpoint that already carries the folded `.weight` (remove_weight_norm) is taken as is.
int effective_weight(fcb_handle* h, const std::string& base, std::vector<int64_t> shape, std::vector<float>* w_out) {
    const HostTensor* w = find(h, base + ".weight");
    if (h->cfg.norm == 0 || w) {
        FCB_TRY(need(h, base + ".weight", shape, &w));
        *w_out = w->data;
        return FCB_OK;
    }
    const HostTensor *g, *v;
    FCB_TRY(need(h, base + ".weight_g", {shape[0], 1, 1}, &g));
    FCB_TRY(need(h, base + ".weight_v", shape, &v));
    const size_t inner = (size_t)(shape[1] * shape[2]);
    w_out->resize(v->data.size());
    for (int64_t i = 0; i < shape[0]; ++i) {
        double ss = 0.0;
        for (size_t j = 0; j < inner; ++j) { const double x = v->data[(size_t)i * inner + j]; ss += x * x; }
        const float f = g->data[(size_t)i] / (float)sqrt(ss);
        for (size_t j = 0; j < inner; ++j) (*w_out)[(size_t)i * inner + j] = v->data[(size_t)i * inner + j] * f;
    }
    return FCB_OK;
}

// GroupNorm(1, C) affine of `norm: time_group_norm`; none for weight_norm / none (get_norm_module returns nn.Identity, conv.py:37-55)
int pack_norm_affine(fcb_handle* h, const std::string& base, int cout, ConvW* o) {
    o->gamma = o->beta = nullptr;
    if (h->cfg.norm != 0) return FCB_OK;
    const HostTensor *g, *be;
    FCB_TRY(need(h, base + ".weight", {cout}, &g));
    FCB_TRY(need(h, base + ".bias", {cout}, &be));
    FCB_TRY(upload(h, g->data, &o->gamma));
    FCB_TRY(upload(h, be->data, &o->beta));
    return FCB_OK;
}

// SConv1d: conv.conv.weight [cout][cin][k] -> [k][cin][cout]
int pack_conv(fcb_handle* h, const std::string& prefix, int cin, int cout, int k, int s, ConvW* o, int dilation = 1) {
    const HostTensor* b;
    std::vector<float> w;
    FCB_TRY(effective_weight(h, prefix + ".conv.conv", {cout, cin, k}, &w));
    FCB_TRY(need(h, prefix + ".conv.conv.bias", {cout}, &b));
    std::vector<float> p((size_t)k * cin * cout);
    for (int co = 0; co < cout; ++co)
        for (int ci = 0; ci < cin; ++ci)
            for (int kk = 0; kk < k; ++kk)
                p[((size_t)kk * cin + ci) * cout + co] = w[((size_t)co * cin + ci) * k + kk];
    o->cin = cin; o->cout = cout; o->k = k; o->s = s; o->d = dilation; o->transposed = false;
    FCB_TRY(pack_tc(h, p, k, cin, cout, o));
    FCB_TRY(upload(h, p, &o->w));
    FCB_TRY(upload(h, b->data, &o->bias));
    FCB_TRY(pack_norm_affine(h, prefix + ".conv.norm", cout, o));
    return FCB_OK;
}

// SConvTranspose1d (k = 2s): convtr.convtr.weight [cin][cout][2s].  out_full[t*s + p] =
//   sum_ci x[t][ci] W[ci][co][p] + x[t-1][ci] W[ci][co][p+s]   (t in [0, T], x[-1] = x[T] = 0)
// == a 2-tap zero-padded conv with C_out' = s*cout whose channels-last output IS out_full[(T+1)*s][cout].
// packed [tap][cin][p*cout + co]: tap 0 <-> x[t-1] (W[..][p+s]), tap 1 <-> x[t] (W[..][p]).
int pack_convtr(fcb_handle* h, const std::string& prefix, int cin, int cout, int s, ConvW* o) {
    const int k = 2 * s;
    const HostTensor* b;
    std::vector<float> w;
    FCB_TRY(effective_weight(h, prefix + ".convtr.convtr", {cin, cout, k}, &w));
    FCB_TRY(need(h, prefix + ".convtr.convtr.bias", {cout}, &b));
    const int ce = s * cout;
    std::vector<float> p((size_t)2 * cin * ce), bias(ce);
    for (int ci = 0; ci < cin; ++ci)
        for (int co = 0; co < cout; ++co)
            for (int ph = 0; ph < s; ++ph) {
                p[((size_t)0 * cin + ci) * ce + ph * cout + co] = w[((size_t)ci * cout + co) * k + ph + s];
                p[((size_t)1 * cin + ci) * ce + ph * cout + co] = w[((size_t)ci * cout + co) * k + ph];
            }
    for (int ph = 0; ph < s; ++ph)
        for (int co = 0; co < cout; ++co) bias[ph * cout + co] = b->data[co];
    o->cin = cin; o->cout = cout; o->k = k; o->s = s; o->transposed = true;
    FCB_TRY(pack_tc(h, p, 2, cin, ce, o));
    FCB_TRY(upload(h, p, &o->w));
    FCB_TRY(upload(h, bias, &o->bias));
    FCB_TRY(pack_norm_affine(h, prefix + ".convtr.norm", cout, o));
    return FCB_OK;
}

// nn.LSTM weights [4H][H] (rows gate-major i,f,g,o) -> [H][4H] with unit-major columns n' = 4*j + gate.
int pack_lstm(fcb_handle* h, const std::string& prefix, int H, int layers, LstmW* o) {
    o->H = H; o->layers = layers;
    for (int l = 0; l < layers; ++l) {
        const HostTensor *wih, *whh, *bih, *bhh;
        const std::string sl = std::to_string(l);
        FCB_TRY(need(h, prefix + ".lstm.weight_ih_l" + sl, {4 * H, H}, &wih));
        FCB_TRY(need(h, prefix + ".lstm.weight_hh_l" + sl, {4 * H, H}, &whh));
        FCB_TRY(need(h, prefix + ".lstm.bias_ih_l" + sl, {4 * H}, &bih));
        FCB_TRY(need(h, prefix + ".lstm.bias_hh_l" + sl, {4 * H}, &bhh));
        std::vector<float> pi((size_t)H * 4 * H), ph((size_t)H * 4 * H), pb(4 * H);
        for (int g = 0; g < 4; ++g)
            for (int j = 0; j < H; ++j) {
                const size_t row = (size_t)g * H + j;
                const size_t col = (size_t)j * 4 + g;
                for (int k = 0; k < H; ++k) {
                    pi[(size_t)k * 4 * H + col] = wih->data[row * H + k];
                    ph[(size_t)k * 4 * H + col] = whh->data[row * H + k];
                }
                pb[col] = bih->data[row] + bhh->data[row];
            }
        ConvW ih;
        ih.cin = H; ih.cout = 4 * H; ih.k = 1; ih.s = 1;
        FCB_TRY(pack_tc(h, pi, 1, H, 4 * H, &ih));
        FCB_TRY(upload(h, pi, &ih.w));
        FCB_TRY(upload(h, pb, &ih.bias));
        float* dwh;
        FCB_TRY(upload(h, ph, &dwh));
        float mx = 0.f;
        for (float v : ph) { const float a = fabsf(v); if (a > mx && a < INFINITY) mx = a; }
        float sc = 1.f;
        if (mx > 0.f) { int e = 0; frexpf(mx, &e); int sh = 14 - e; if (sh > 40) sh = 40; if (sh < -40) sh = -40; sc = ldexpf(1.f, sh); }
        o->ih.push_back(ih); o->whh.push_back(dwh); o->whh_scale.push_back(sc);
    }
    return FCB_OK;
}

int pack_resblock(fcb_handle* h, const std::string& prefix, int dim, ResBlockW* o, int dilation = 1) {
    FCB_TRY(pack_conv(h, prefix + ".block.1", dim, dim / 2, h->cfg.residual_kernel_size, 1, &o->c1, dilation));
    FCB_TRY(pack_conv(h, prefix + ".block.3", dim / 2, dim, 1, 1, &o->c2));
    FCB_TRY(pack_conv(h, prefix + ".shortcut", dim, dim, 1, 1, &o->sc));
    return FCB_OK;
}

// ------------------------------------------------------------------------------------------- run helpers
// One API call.  Every temporary comes from the stream-ordered pool through pool_alloc and is tracked here, so an
// early return on an error path cannot leak: whatever is still live is returned to the pool by the destructor.
struct Run {
    fcb_handle* h;
    int B;
    cudaStream_t st;
    int phase = -1;
    std::vector<void*> live;
    Run(fcb_handle* h_, int B_, cudaStream_t st_) : h(h_), B(B_), st(st_) {}
    Run(const Run&) = delete;
    Run& operator=(const Run&) = delete;
    ~Run() {
        for (void* p : live) cudaFreeAsync(p, st);
    }
};

int pool_alloc(Run& r, void** p, size_t bytes) {
    fcb_handle* h = r.h;
    FCB_CK(cudaMallocAsync(p, bytes, r.st));
    r.live.push_back(*p);
    return FCB_OK;
}

int pool_free(Run& r, void* p) {
    fcb_handle* h = r.h;
    if (!p) return FCB_OK;
    for (size_t i = 0; i < r.live.size(); ++i)
        if (r.live[i] == p) { r.live[i] = r.live.back(); r.live.pop_back(); break; }
    FCB_CK(cudaFreeAsync(p, r.st));
    return FCB_OK;
}

int alloc_f(Run& r, float** p, size_t n) { return pool_alloc(r, (void**)p, n * sizeof(float)); }

int release(Run& r, Act& a) {
    fcb_handle* h = r.h;
    if (a.owned) {
        FCB_TRY(pool_free(r, a.p));
        FCB_TRY(pool_free(r, a.stats));
        FCB_TRY(pool_free(r, a.coef));
    }
    a = Act();
    return FCB_OK;
}

int phase_begin(Run& r, int ph) {
    fcb_handle* h = r.h;
    if (!h->profiling) return FCB_OK;
    r.phase = ph;
    h->ev_used[ph] = true;
    FCB_CK(cudaEventRecord(h->ev[ph][0], r.st));
    return FCB_OK;
}
int phase_end(Run& r) {
    fcb_handle* h = r.h;
    if (!h->profiling || r.phase < 0) return FCB_OK;
    FCB_CK(cudaEventRecord(h->ev[r.phase][1], r.st));
    r.phase = -1;
    return FCB_OK;
}

InView view_of(const Act& a) {
    InView v;
    v.x = a.p; v.stats = a.stats; v.gamma = a.gamma; v.beta = a.beta; v.coef = a.coef;
    v.clip_stride = a.clip_stride; v.row_off = a.row_off;
    return v;
}

// One SConv1d / SConvTranspose1d / 1x1 GEMM.  in1 may be null.  want_norm=false -> plain output (LSTM input
// projection).  Dispatch: tensor-core implicit GEMM (conv_tc.cu) when the layer has a TC weight image and the
// input needs no division prologue, else the fp32 SIMT kernel (conv_simt.cu).
int run_conv(Run& r, const Act& in0, const Act* in1, bool elu, const float* div_scale, const ConvW& L,
             bool want_norm, Act* out) {
    fcb_handle* h = r.h;
    want_norm = want_norm && L.gamma != nullptr;   // norm: weight_norm / none -> the conv output is the layer output
    const bool causal = h->cfg.causal != 0;
    ConvParams p{};
    p.in0 = view_of(in0);
    if (in1) p.in1 = view_of(*in1); else p.in1.x = nullptr;
    p.div_scale = div_scale;
    p.elu = elu ? 1 : 0;
    p.T_in = in0.T; p.C_in = in0.C;
    p.in_ch_stride = in0.ch_stride;
    if (in0.C != L.cin) return fail(h, FCB_E_INVALID, "internal: channel mismatch");
    Act o;
    if (!L.transposed) {
        const int k = L.k, s = L.s, d = L.d;
        const int padding_total = (k - 1) * d - (s - 1);
        // get_extra_padding_for_conv1d (conv.py:57-64), integer form of ceil((T - k + pt)/s)
        const int num = in0.T - ((k - 1) * d + 1) + padding_total;     // effective kernel size (k - 1) * d + 1 (conv.py:57-64)
        const int n_frames_ceil = (num >= 0 ? (num + s - 1) / s : -((-num) / s)) + 1;
        const int ideal = (n_frames_ceil - 1) * s + ((k - 1) * d + 1 - padding_total);
        const int extra = ideal - in0.T;
        // causal: pad1d(x, (padding_total, extra_padding)) (conv.py:251-253), else the asymmetric split (:255-258)
        const int pr = causal ? 0 : padding_total / 2, pl = padding_total - pr;
        const int pr_tot = pr + extra;
        const int max_pad = pl > pr_tot ? pl : pr_tot;
        p.K = k; p.S = s; p.D = d; p.pad_l = pl; p.pad_zero = 0;
        p.T_ext = in0.T <= max_pad ? max_pad + 1 : in0.T;     // pad1d tiny-input branch (conv.py:89-97)
        p.T_out = (in0.T + pl + pr_tot - ((k - 1) * d + 1)) / s + 1;
        p.C_out = L.cout;
        o.T = p.T_out; o.C = L.cout; o.clip_stride = (long long)p.T_out * L.cout; o.row_off = 0;
    } else {
        const int s = L.s;
        p.K = 2; p.S = 1; p.D = 1; p.pad_l = 1; p.pad_zero = 1; p.T_ext = in0.T;
        p.T_out = in0.T + 1;
        p.C_out = s * L.cout;
        const int padding_total = L.k - s;                    // conv.py:283-303
        // causal (trim_right_ratio = 1): everything is trimmed on the right (conv.py:293-297)
        const int pr = causal ? padding_total : padding_total / 2, pl = padding_total - pr;
        o.T = in0.T * s; o.C = L.cout; o.clip_stride = (long long)p.T_out * p.C_out; o.row_off = pl;
    }
    p.w = L.w; p.bias = L.bias; p.w_tc = L.w_tc; p.n_tile = L.n_tile; p.tc_w_scale = L.tc_scale;
    p.out_clip_stride = (long long)p.T_out * p.C_out;
    const bool tc = h->use_tc && L.n_tile > 0 && L.w_tc && !div_scale && !in0.ch_stride;
    FCB_TRY(alloc_f(r, &o.p, (size_t)r.B * p.out_clip_stride));
    o.owned = true;
    p.out = o.p;
    double* partials = nullptr;
    const bool c1 = !tc && conv_cout1_supported(p);
    const int nparts = tc ? conv_tc_num_parts(p.T_out, p.C_out)
                          : (c1 ? conv_cout1_num_parts(p.T_out, p.C_out) : conv_num_parts(p.T_out, p.C_out, p.C_in, p.K, r.B));
    if (want_norm) {
        FCB_TRY(pool_alloc(r, (void**)&partials, (size_t)r.B * nparts * 2 * sizeof(double)));
        FCB_TRY(alloc_f(r, &o.stats, (size_t)r.B * 2));
        FCB_TRY(alloc_f(r, &o.coef, (size_t)r.B * 2 * o.C));
        o.gamma = L.gamma; o.beta = L.beta;
    }
    p.partials = partials;
    int np2 = 0;
    if (tc) FCB_CK(launch_conv_tc(p, r.B, r.st, &np2));
    else if (c1) FCB_CK(launch_conv_cout1(p, r.B, r.st, &np2));
    else FCB_CK(launch_conv(p, r.B, r.st, &np2));
    h->launches++;
    if (want_norm) {
        if (np2 != nparts) return fail(h, FCB_E_INVALID, "internal: partial count mismatch");
        FCB_CK(launch_stats_finalize(partials, nparts, (double)p.T_out * p.C_out, h->cfg.gn_eps, 0, o.stats, r.B, r.st,
                                     L.gamma, L.beta, o.C, o.coef));
        h->launches++;
        FCB_TRY(pool_free(r, partials));
    }
    *out = o;
    return FCB_OK;
}

// SLSTM (lstm.py:22-28): y = LSTM(x) + x.  x is a normalised view; y is a plain tensor.
int run_lstm(Run& r, const Act& x, const LstmW& W, Act* out) {
    fcb_handle* h = r.h;
    const int H = W.H, T = x.T, B = r.B;
    if (x.C != H) return fail(h, FCB_E_INVALID, "internal: lstm width mismatch");
    if (lstm_pick_units(H) == 0) return fail(h, FCB_E_INVALID, "lstm width not supported (needs H % 4 == 0 and the W_hh slice to fit shared memory)");
    Act cur = x;       // not owned copy semantics: only release what we allocate
    cur.owned = false;
    Act y;
    for (int l = 0; l < W.layers; ++l) {
        Act gx;
        FCB_TRY(run_conv(r, cur, nullptr, false, nullptr, W.ih[l], false, &gx));
        Act hs;
        FCB_TRY(alloc_f(r, &hs.p, (size_t)B * T * H));
        hs.owned = true; hs.T = T; hs.C = H; hs.clip_stride = (long long)T * H;
        const bool last = (l == W.layers - 1);
        if (last) {
            FCB_TRY(alloc_f(r, &y.p, (size_t)B * T * H));
            y.owned = true; y.T = T; y.C = H; y.clip_stride = (long long)T * H;
        }
        LstmSeqParams sp{};
        sp.gx = gx.p; sp.whh = W.whh[l]; sp.h_seq = hs.p;
        sp.y_out = last ? y.p : nullptr;
        sp.skip = view_of(x);
        sp.barrier = h->lstm_barrier;
        sp.trace = h->lstm_trace;
        sp.whh_scale = W.whh_scale[l];
        sp.whh_inv_scale = 1.0f / (W.whh_scale[l] * 4096.0f);
        sp.B = B; sp.T = T; sp.H = H;
        FCB_CK(launch_lstm_seq(sp, r.st));
        h->launches += 1;
        FCB_TRY(release(r, gx));
        if (l > 0) FCB_TRY(release(r, cur));
        cur = hs;
    }
    FCB_TRY(release(r, cur));
    *out = y;
    return FCB_OK;
}

// x (+ x1: the input may itself be the pending sum shortcut + block of the previous resblock of the stage)
int run_resblock(Run& r, const Act& x, const ResBlockW& W, Act* sc_out, Act* blk_out, const Act* x1 = nullptr) {
    Act h1, h2, sc;
    FCB_TRY(run_conv(r, x, x1, true, nullptr, W.c1, true, &h1));
    FCB_TRY(run_conv(r, h1, nullptr, true, nullptr, W.c2, true, &h2));
    FCB_TRY(release(r, h1));
    FCB_TRY(run_conv(r, x, x1, false, nullptr, W.sc, true, &sc));
    *sc_out = sc; *blk_out = h2;
    return FCB_OK;
}

// Encodec._encode_frame (codec_basic.py:361-380) + SEANetEncoder.forward; returns the final conv's raw
// output view (GroupNorm deferred into the RVQ kernel's load).  wav is [B][L], or channel-planar [B][2][L] for a stereo
// handle: the scale comes from the mono mix and the first conv reads both channel rows directly.
int run_encoder(Run& r, const float* wav, int L, float* scale_out, Act* out) {
    fcb_handle* h = r.h;
    const int B = r.B, C = h->channels();
    FCB_TRY(phase_begin(r, FCB_PHASE_ENCODER_CONV));
    float* scale = nullptr;
    bool scale_owned = false;
    if (h->cfg.audio_normalize) {
        double* partials = nullptr;
        int nparts = sumsq_num_parts(L), np2 = 0;
        FCB_TRY(pool_alloc(r, (void**)&partials, (size_t)B * nparts * 2 * sizeof(double)));
        if (scale_out) scale = scale_out; else { FCB_TRY(alloc_f(r, &scale, B)); scale_owned = true; }
        FCB_CK(launch_sumsq_partials(wav, B, L, partials, &np2, r.st, C));
        FCB_CK(launch_stats_finalize(partials, nparts, (double)L, 0.f, 1, scale, B, r.st));
        h->launches += 2;
        FCB_TRY(pool_free(r, partials));
    } else if (scale_out) {
        FCB_CK(launch_fill(scale_out, 1.0f, B, r.st));
        h->launches++;
    }
    Act x;
    x.p = const_cast<float*>(wav); x.T = L; x.C = C; x.clip_stride = (long long)C * L;
    if (C > 1) x.ch_stride = L;
    Act a;
    FCB_TRY(run_conv(r, x, nullptr, false, scale, h->enc_conv0, true, &a));
    if (scale_owned) FCB_TRY(pool_free(r, scale));
    const int nres = (int)(h->enc_rb.size() / (h->enc_down.empty() ? 1 : h->enc_down.size()));
    for (size_t i = 0; i < h->enc_down.size(); ++i) {
        Act sc, blk, d;
        FCB_TRY(run_resblock(r, a, h->enc_rb[i * nres], &sc, &blk));
        FCB_TRY(release(r, a));
        for (int j = 1; j < nres; ++j) {          // stacked residual blocks: the next block consumes the pending sum
            Act sc2, blk2;
            FCB_TRY(run_resblock(r, sc, h->enc_rb[i * nres + j], &sc2, &blk2, &blk));
            FCB_TRY(release(r, sc));
            FCB_TRY(release(r, blk));
            sc = sc2; blk = blk2;
        }
        FCB_TRY(run_conv(r, sc, &blk, true, nullptr, h->enc_down[i], true, &d));
        FCB_TRY(release(r, sc));
        FCB_TRY(release(r, blk));
        a = d;
    }
    FCB_TRY(phase_end(r));
    // phase ENCODER_LSTM = SLSTM + the final k7 conv (both live at T' frames)
    FCB_TRY(phase_begin(r, FCB_PHASE_ENCODER_LSTM));
    if (h->cfg.lstm_layers > 0) {
        Act y;
        FCB_TRY(run_lstm(r, a, h->enc_lstm, &y));
        FCB_TRY(release(r, a));
        a = y;
    }
    Act f;
    FCB_TRY(run_conv(r, a, nullptr, true, nullptr, h->enc_final, true, &f));
    FCB_TRY(release(r, a));
    FCB_TRY(phase_end(r));
    *out = f;
    return FCB_OK;
}

// SEANetDecoder.forward + Encodec._decode_frame (codec_basic.py:398-408) + trim (:711).
int run_decoder_freq(Run& r, const float* emb, int n_frames, const float* scale, float* wav_out, int out_len);
int run_plain_tc(Run& r, const float* x, int T_in, const ConvW& L, int T_out, float* out);
int pack_stft_bases(fcb_handle* h);

int run_decoder_time(Run& r, const float* emb, int n_frames, const float* scale, float* wav_out, int out_len) {
    fcb_handle* h = r.h;
    const int hop = h->hop();
    if (out_len > n_frames * hop || out_len <= 0) return fail(h, FCB_E_INVALID, "out_len must be in (0, T'*hop]");
    if (r.B > 512) return fail(h, FCB_E_INVALID, "decode: at most 512 clips per call (split the batch)");
    Act e;
    e.p = const_cast<float*>(emb); e.T = n_frames; e.C = h->cfg.dimension; e.clip_stride = (long long)n_frames * e.C;
    FCB_TRY(phase_begin(r, FCB_PHASE_DECODER_LSTM));
    Act a;
    FCB_TRY(run_conv(r, e, nullptr, false, nullptr, h->dec_conv0, true, &a));
    if (h->cfg.lstm_layers > 0) {
        Act y;
        FCB_TRY(run_lstm(r, a, h->dec_lstm, &y));
        FCB_TRY(release(r, a));
        a = y;
    }
    FCB_TRY(phase_end(r));
    FCB_TRY(phase_begin(r, FCB_PHASE_DECODER_CONV));
    Act sc = a, blk;   // "sc + blk" is the current tensor; blk unused before the first resblock
    bool have_blk = false;
    for (size_t i = 0; i < h->dec_up.size(); ++i) {
        Act u;
        FCB_TRY(run_conv(r, sc, have_blk ? &blk : nullptr, true, nullptr, h->dec_up[i], true, &u));
        FCB_TRY(release(r, sc));
        if (have_blk) FCB_TRY(release(r, blk));
        const int nres = (int)(h->dec_rb.size() / h->dec_up.size());
        FCB_TRY(run_resblock(r, u, h->dec_rb[i * nres], &sc, &blk));
        FCB_TRY(release(r, u));
        for (int j = 1; j < nres; ++j) {
            Act sc2, blk2;
            FCB_TRY(run_resblock(r, sc, h->dec_rb[i * nres + j], &sc2, &blk2, &blk));
            FCB_TRY(release(r, sc));
            FCB_TRY(release(r, blk));
            sc = sc2; blk = blk2;
        }
        have_blk = true;
    }
    Act f;
    FCB_TRY(run_conv(r, sc, have_blk ? &blk : nullptr, true, nullptr, h->dec_final, true, &f));
    FCB_TRY(release(r, sc));
    if (have_blk) FCB_TRY(release(r, blk));
    FCB_CK(launch_final_output(f.p, f.stats, f.gamma, f.beta, scale, r.B, f.T, out_len, wav_out, r.st, f.C));
    h->launches++;
    FCB_TRY(release(r, f));
    FCB_TRY(phase_end(r));
    return FCB_OK;
}

// =============================================================================================== FreqCodec (arch 1)
typedef fcb_handle::Conv2W Conv2W;
typedef fcb_handle::ResBlock2W ResBlock2W;

// Tensor-core image of a packed 2-D layer wp = [kt][kf*cin][cout_eff] (the 1-D slab format with C_in = kf*cin gathered
// channels); C_out_eff is zero-padded to a multiple of 16 (the 32 -> 3 output conv), bias alike.
int pack_tc2d(fcb_handle* h, const std::vector<float>& wp, const std::vector<float>& bias, int cout_eff, Conv2W* o) {
    o->n_tile = 0; o->tc_class = 0;
    const int ck = o->kf_eff * o->cin, kt = o->kt_eff;
    const int cout_tc = (cout_eff + 15) / 16 * 16;
    if (!h->use_tc || !conv_tc_supported_2d(o->cin, cout_tc, kt, o->transposed ? 1 : o->st)) return FCB_OK;
    if (cout_tc != cout_eff && o->transposed) return FCB_OK;
    std::vector<float> img;
    const int n_tile = conv_tc_n_tile(cout_tc);
    if (cout_tc == cout_eff) {
        build_tc_image_f16(wp, kt, ck, cout_eff, n_tile, &img, &o->tc_scale);
        o->bias_tc = nullptr;
    } else {
        std::vector<float> wpad((size_t)kt * ck * cout_tc, 0.f), bpad(cout_tc, 0.f);
        for (size_t r = 0; r < (size_t)kt * ck; ++r)
            for (int co = 0; co < cout_eff; ++co) wpad[r * cout_tc + co] = wp[r * cout_eff + co];
        for (int co = 0; co < cout_eff; ++co) bpad[co] = bias[co];
        build_tc_image_f16(wpad, kt, ck, cout_tc, n_tile, &img, &o->tc_scale);
        FCB_TRY(upload(h, bpad, &o->bias_tc));
    }
    FCB_TRY(upload(h, img, &o->w_tc));
    o->n_tile = n_tile; o->cout_tc = cout_tc;
    o->tc_class = cout_tc != cout_eff ? 4 : (o->cin % 32 == 0 ? 1 : 2);
    return FCB_OK;
}

// SConv2d weight [cout][cin][kf][kt] -> [kt][kf*cin_store + ci][cout]; cin_store >= cin pads the stored input channels
// with zero weights (the 3-channel mag_phase features are kept as 4 channels so that a frequency tap is one 16-byte load).
// groups > 1 (conv_group_ratio): the reference weight is [cout][cin / groups][kf][kt]; it is expanded into the dense
// block-diagonal matrix (zeros outside the groups), so the same dense kernels run it -- identical results, dense MACs.
int pack_conv2d(fcb_handle* h, const std::string& prefix, int cin, int cout, int kf, int kt, int sf, int st, Conv2W* o,
                int cin_store = 0, int groups = 1) {
    if (cin_store < cin) cin_store = cin;
    if (groups < 1 || cin % groups != 0 || cout % groups != 0)
        return fail(h, FCB_E_INVALID, "conv groups do not divide the channels of " + prefix + " (check conv_group_ratio)");
    const int cig = cin / groups, cog = cout / groups;
    const HostTensor *w, *b, *g, *be;
    FCB_TRY(need(h, prefix + ".conv.conv.weight", {cout, cig, kf, kt}, &w));
    FCB_TRY(need(h, prefix + ".conv.conv.bias", {cout}, &b));
    FCB_TRY(need(h, prefix + ".conv.norm.weight", {cout}, &g));
    FCB_TRY(need(h, prefix + ".conv.norm.bias", {cout}, &be));
    std::vector<float> p((size_t)kt * kf * cin_store * cout, 0.f);
    for (int co = 0; co < cout; ++co) {
        const int ci0 = (co / cog) * cig;                 // first input channel of this output channel's group
        for (int cl = 0; cl < cig; ++cl)
            for (int a = 0; a < kf; ++a)
                for (int c = 0; c < kt; ++c)
                    p[(((size_t)c * kf + a) * cin_store + ci0 + cl) * cout + co] = w->data[(((size_t)co * cig + cl) * kf + a) * kt + c];
    }
    o->cin = cin_store; o->cout = cout; o->kf = kf; o->kt = kt; o->sf = sf; o->st = st; o->transposed = false;
    o->kf_eff = kf; o->kt_eff = kt;
    FCB_TRY(upload(h, p, &o->w));
    FCB_TRY(upload(h, b->data, &o->bias));
    FCB_TRY(upload(h, g->data, &o->gamma));
    FCB_TRY(upload(h, be->data, &o->beta));
    FCB_TRY(pack_tc2d(h, p, b->data, cout, o));
    return FCB_OK;
}

// SConvTranspose2d (k = 2s per axis) weight [cin][cout][2fr][2tr] -> 2x2-tap conv, C_out' = fr*tr*cout:
// packed[kti][kfi*cin + ci][(pf*tr + pt)*cout + co] = W[ci][co][pf + (1-kfi)*fr][pt + (1-kti)*tr]
// (tap index 0 <-> the previous input row / column, as in pack_convtr).
int pack_convtr2d(fcb_handle* h, const std::string& prefix, int cin, int cout, int fr, int tr, Conv2W* o, int groups = 1) {
    const int kf = 2 * fr, kt = 2 * tr;
    if (groups < 1 || cin % groups != 0 || cout % groups != 0)
        return fail(h, FCB_E_INVALID, "conv groups do not divide the channels of " + prefix + " (check tr_conv_group_ratio)");
    const int cig = cin / groups, cog = cout / groups;     // nn.ConvTranspose2d weight: [cin][cout / groups][kf][kt]
    const HostTensor *w, *b, *g, *be;
    FCB_TRY(need(h, prefix + ".convtr.convtr.weight", {cin, cog, kf, kt}, &w));
    FCB_TRY(need(h, prefix + ".convtr.convtr.bias", {cout}, &b));
    FCB_TRY(need(h, prefix + ".convtr.norm.weight", {cout}, &g));
    FCB_TRY(need(h, prefix + ".convtr.norm.bias", {cout}, &be));
    const int ce = fr * tr * cout;
    std::vector<float> p((size_t)2 * 2 * cin * ce, 0.f), bias(ce);
    for (int kti = 0; kti < 2; ++kti)
        for (int kfi = 0; kfi < 2; ++kfi)
            for (int ci = 0; ci < cin; ++ci)
                for (int pf = 0; pf < fr; ++pf)
                    for (int pt = 0; pt < tr; ++pt)
                        for (int cl = 0; cl < cog; ++cl) {
                            const int co = (ci / cig) * cog + cl;      // output channels of input channel ci's group
                            p[(((size_t)kti * 2 + kfi) * cin + ci) * ce + (pf * tr + pt) * cout + co] =
                                w->data[(((size_t)ci * cog + cl) * kf + pf + (1 - kfi) * fr) * kt + pt + (1 - kti) * tr];
                        }
    for (int ph = 0; ph < fr * tr; ++ph)
        for (int co = 0; co < cout; ++co) bias[ph * cout + co] = b->data[co];
    o->cin = cin; o->cout = cout; o->kf = kf; o->kt = kt; o->sf = fr; o->st = tr; o->transposed = true;
    o->kf_eff = 2; o->kt_eff = 2;
    FCB_TRY(upload(h, p, &o->w));
    FCB_TRY(upload(h, bias, &o->bias));
    FCB_TRY(upload(h, g->data, &o->gamma));
    FCB_TRY(upload(h, be->data, &o->beta));
    FCB_TRY(pack_tc2d(h, p, bias, ce, o));
    return FCB_OK;
}

// groups = channels // 2 // ratio (seanet_encoder.py:224,234,321; seanet_decoder.py:324), dense when ratio <= 0
int conv_groups_of(int channels, int ratio) { return ratio > 0 ? channels / 2 / ratio : 1; }

int pack_resblock2d(fcb_handle* h, const std::string& prefix, int dim, ResBlock2W* o) {
    const int rk = h->cfg.residual_kernel_size, gr = h->cfg.conv_group_ratio;
    const int gb = conv_groups_of(dim / 2, gr);            // min(in, out) = dim / 2 for both block convs
    FCB_TRY(pack_conv2d(h, prefix + ".block.1", dim, dim / 2, rk, rk, 1, 1, &o->c1, 0, gb));
    FCB_TRY(pack_conv2d(h, prefix + ".block.3", dim / 2, dim, 1, 1, 1, 1, &o->c2, 0, gb));
    FCB_TRY(pack_conv2d(h, prefix + ".shortcut", dim, dim, 1, 1, 1, 1, &o->sc, 0, conv_groups_of(dim, gr)));
    return FCB_OK;
}

// A raw 2-D activation [B][F_raw][T_raw][C] plus its deferred GroupNorm and logical window.
struct Act2 {
    float* p = nullptr;
    int F_raw = 0, T_raw = 0, f_off = 0, t_off = 0;
    int F = 0, T = 0, C = 0;
    float* stats = nullptr;
    float* coef = nullptr;
    const float* gamma = nullptr;
    const float* beta = nullptr;
    bool owned = false;
};

int release2(Run& r, Act2& a) {
    if (a.owned) {
        FCB_TRY(pool_free(r, a.p));
        FCB_TRY(pool_free(r, a.stats));
        FCB_TRY(pool_free(r, a.coef));
    }
    a = Act2();
    return FCB_OK;
}

InView2 view2_of(const Act2& a) {
    InView2 v;
    v.x = a.p; v.coef = a.coef; v.F_raw = a.F_raw; v.T_raw = a.T_raw; v.f_off = a.f_off; v.t_off = a.t_off;
    return v;
}

// SConv2d / SConvTranspose2d (non-causal).
int run_conv2d(Run& r, const Act2& in0, const Act2* in1, bool elu, const Conv2W& L, Act2* out) {
    fcb_handle* h = r.h;
    if (in0.C != L.cin) return fail(h, FCB_E_INVALID, "internal: 2-D channel mismatch");
    Conv2dParams p{};
    p.in0 = view2_of(in0);
    if (in1) p.in1 = view2_of(*in1); else p.in1.x = nullptr;
    p.elu = elu ? 1 : 0;
    p.B = r.B; p.F_in = in0.F; p.T_in = in0.T; p.C_in = in0.C;
    p.w = L.w; p.bias = L.bias;
    Act2 o;
    if (!L.transposed) {
        const int pt_f = (L.kf - 1) - (L.sf - 1), pt_t = (L.kt - 1) - (L.st - 1);
        const int num = in0.T - L.kt + pt_t;
        const int n_frames_ceil = (num >= 0 ? (num + L.st - 1) / L.st : -((-num) / L.st)) + 1;
        const int extra = (n_frames_ceil - 1) * L.st + (L.kt - pt_t) - in0.T;
        const int f_after = pt_f / 2, f_before = pt_f - f_after;
        const int t_after = pt_t / 2, t_before = pt_t - t_after + extra;     // extra on the LEFT in 2-D (conv.py:368)
        if (in0.F <= (f_before > f_after ? f_before : f_after) || in0.T <= (t_before > t_after ? t_before : t_after))
            return fail(h, FCB_E_INVALID, "2-D conv: input smaller than its reflect padding is not supported");
        p.KF = L.kf; p.KT = L.kt; p.SF = L.sf; p.ST = L.st; p.pad_f = f_before; p.pad_t = t_before; p.pad_zero = 0;
        p.F_out = (in0.F + pt_f - L.kf) / L.sf + 1;
        p.T_out = (in0.T + pt_t + extra - L.kt) / L.st + 1;
        p.C_out_eff = L.cout; p.FR = 1; p.TR = 1; p.Cc = L.cout;
        o.F_raw = o.F = p.F_out; o.T_raw = o.T = p.T_out;
    } else {
        const int fr = L.sf, tr = L.st;
        p.KF = 2; p.KT = 2; p.SF = 1; p.ST = 1; p.pad_f = 1; p.pad_t = 1; p.pad_zero = 1;
        p.F_out = in0.F + 1; p.T_out = in0.T + 1;
        p.C_out_eff = fr * tr * L.cout; p.FR = fr; p.TR = tr; p.Cc = L.cout;
        o.F_raw = p.F_out * fr; o.T_raw = p.T_out * tr;
        const int pf = L.kf - fr, ptt = L.kt - tr;                            // conv.py:410-445
        const int pf_r = pf / 2, pf_l = pf - pf_r, pt_r = ptt / 2, pt_l = ptt - pt_r;
        const int fo_l = L.out_pad[0][0], fo_r = L.out_pad[0][1], to_l = L.out_pad[1][0], to_r = L.out_pad[1][1];
        const int fl = pf_l - fo_l > 0 ? pf_l - fo_l : 0, frr = pf_r - fo_r > 0 ? pf_r - fo_r : 0;
        const int tl = pt_l - to_l > 0 ? pt_l - to_l : 0, trr = pt_r - to_r > 0 ? pt_r - to_r : 0;
        o.f_off = fl; o.t_off = tl;
        o.F = o.F_raw - fl - frr; o.T = o.T_raw - tl - trr;
    }
    o.C = L.cout;
    const size_t per_clip = (size_t)o.F_raw * o.T_raw * o.C;
    FCB_TRY(alloc_f(r, &o.p, (size_t)r.B * per_clip));
    o.owned = true;
    p.out = o.p;
    // tensor-core path (conv_tc.cu, 2-D mode) when the layer has a slab image and its class is enabled
    // halo-tile SIMT kernel for C_out <= 4 (the 32 -> 3 output conv), "conv2d_small_cout" option (default on)
    const bool small = h->conv2d_small_cout && !L.transposed && conv2d_small_cout_supported(p);
    const bool tc = !small && h->use_tc && L.n_tile > 0 && L.w_tc && (h->use_tc2d & L.tc_class) != 0;
    // statistics partials per clip: the pseudo-clip kernels emit n per output frequency row
    const int nparts = small ? conv2d_small_cout_num_parts(p)
                             : p.F_out * (tc ? conv_tc_num_parts(p.T_out, L.cout_tc) : conv2d_num_parts(p));
    double* partials = nullptr;
    FCB_TRY(pool_alloc(r, (void**)&partials, (size_t)r.B * nparts * 2 * sizeof(double)));
    FCB_TRY(alloc_f(r, &o.stats, (size_t)r.B * 2));
    FCB_TRY(alloc_f(r, &o.coef, (size_t)r.B * 2 * o.C));
    o.gamma = L.gamma; o.beta = L.beta;
    p.partials = partials;
    if (tc) {
        ConvParams q{};
        q.in0.x = in0.p; q.in0.coef = in0.coef; q.in0.row_off = in0.t_off;
        q.in0.clip_stride = (long long)in0.F_raw * in0.T_raw * in0.C;
        if (in1) {
            q.in1.x = in1->p; q.in1.coef = in1->coef; q.in1.row_off = in1->t_off;
            q.in1.clip_stride = (long long)in1->F_raw * in1->T_raw * in1->C;
        }
        q.elu = p.elu;
        q.T_in = in0.T; q.C_in = p.KF * in0.C;
        q.K = p.KT; q.S = p.ST; q.D = 1; q.pad_l = p.pad_t; q.T_ext = in0.T; q.pad_zero = p.pad_zero;
        q.w_tc = L.w_tc; q.n_tile = L.n_tile; q.tc_w_scale = L.tc_scale; q.bias = L.bias_tc ? L.bias_tc : L.bias;
        q.out = o.p; q.T_out = p.T_out; q.C_out = L.cout_tc;
        q.out_clip_stride = (long long)p.T_out * L.cout_tc;
        q.partials = partials;
        q.fq.KF = p.KF; q.fq.SF = p.SF; q.fq.pad_f = p.pad_f; q.fq.F_in = in0.F; q.fq.F_out = p.F_out; q.fq.cin = in0.C;
        q.fq.T_raw0 = in0.T_raw; q.fq.f_off0 = in0.f_off;
        q.fq.T_raw1 = in1 ? in1->T_raw : 0; q.fq.f_off1 = in1 ? in1->f_off : 0;
        q.fq.FR = p.FR; q.fq.TR = p.TR;
        q.fq.Cc = L.tc_class == 4 ? L.cout_tc : p.Cc;      // padded image: one phase of cout_tc columns, Cc real ones stored
        q.fq.c_store = p.Cc;
        int np2 = 0;
        FCB_CK(launch_conv_tc(q, r.B * p.F_out, r.st, &np2));
        if (np2 * p.F_out != nparts) return fail(h, FCB_E_INVALID, "internal: partial count mismatch (2-D)");
    } else if (small) {
        FCB_CK(launch_conv2d_small_cout(p, r.st));
    } else {
        FCB_CK(launch_conv2d(p, r.st));
    }
    FCB_CK(launch_stats_finalize(partials, nparts, (double)per_clip, h->cfg.gn_eps, 0, o.stats, r.B, r.st, L.gamma,
                                 L.beta, o.C, o.coef));
    h->launches += 2;
    FCB_TRY(pool_free(r, partials));
    *out = o;
    return FCB_OK;
}

int run_resblock2d(Run& r, const Act2& x, const ResBlock2W& W, Act2* sc_out, Act2* blk_out) {
    Act2 h1, h2, sc;
    FCB_TRY(run_conv2d(r, x, nullptr, true, W.c1, &h1));
    FCB_TRY(run_conv2d(r, h1, nullptr, true, W.c2, &h2));
    FCB_TRY(release2(r, h1));
    FCB_TRY(run_conv2d(r, x, nullptr, false, W.sc, &sc));
    *sc_out = sc; *blk_out = h2;
    return FCB_OK;
}

int stft_frames(const fcb_handle* h, int L) { return 1 + L / h->cfg.stft_hop; }

// FreqCodec._encode_frame (mag_phase) + SEANetEncoder2d.forward; returns the final conv1d's raw output view.
int run_encoder_freq(Run& r, const float* wav, int L, float* scale_out, Act* out) {
    fcb_handle* h = r.h;
    const int B = r.B;
    const fcb_config& c = h->cfg;
    if (L <= c.n_fft / 2) return fail(h, FCB_E_INVALID, "clip shorter than n_fft/2 (reflect padding of the STFT)");
    FCB_TRY(phase_begin(r, FCB_PHASE_ENCODER_CONV));
    float* scale = nullptr;
    bool scale_owned = false;
    if (c.audio_normalize) {
        double* partials = nullptr;
        int nparts = sumsq_num_parts(L), np2 = 0;
        FCB_TRY(pool_alloc(r, (void**)&partials, (size_t)B * nparts * 2 * sizeof(double)));
        if (scale_out) scale = scale_out; else { FCB_TRY(alloc_f(r, &scale, B)); scale_owned = true; }
        FCB_CK(launch_sumsq_partials(wav, B, L, partials, &np2, r.st));
        FCB_CK(launch_stats_finalize(partials, nparts, (double)L, 0.f, 1, scale, B, r.st));
        h->launches += 2;
        FCB_TRY(pool_free(r, partials));
    } else if (scale_out) {
        FCB_CK(launch_fill(scale_out, 1.0f, B, r.st));
        h->launches++;
    }
    const int n_bins = c.n_fft / 2 + 1, Ts = stft_frames(h, L);
    Act2 a;
    const int cfe = h->f_enc_conv0.cin;                 // 3 mag_phase features stored as 4 channels (pack_conv2d)
    FCB_TRY(alloc_f(r, &a.p, (size_t)B * n_bins * Ts * cfe));
    a.owned = true; a.F_raw = a.F = n_bins; a.T_raw = a.T = Ts; a.C = cfe;
    if (h->stft_tc && !h->stft_packed) { h->stft_packed = true; FCB_TRY(pack_stft_bases(h)); }   // lazily: the default path never builds them
    if (h->stft_tc && h->stft_w.n_tile > 0) {       // rows of 32 samples -> DFT-basis GEMM -> mag_phase features
        const int n_rows = (L + c.n_fft + 31) / 32;
        float *rows = nullptr, *spec = nullptr;
        FCB_TRY(alloc_f(r, &rows, (size_t)B * n_rows * 32));
        FCB_TRY(alloc_f(r, &spec, (size_t)B * Ts * h->stft_ld));
        FCB_CK(launch_wave_rows(wav, scale, B, L, c.n_fft, n_rows, rows, r.st));
        FCB_TRY(run_plain_tc(r, rows, n_rows, h->stft_w, Ts, spec));
        FCB_CK(launch_magphase_from_spec(spec, h->stft_ld, B, n_bins, Ts, cfe, a.p, r.st));
        h->launches += 2;
        FCB_TRY(pool_free(r, rows));
        FCB_TRY(pool_free(r, spec));
    } else {
        FCB_CK(launch_stft_magphase(wav, scale, B, L, c.n_fft, c.stft_hop, Ts, cfe, a.p, r.st));
        h->launches++;
    }
    if (scale_owned) FCB_TRY(pool_free(r, scale));
    Act2 x;
    FCB_TRY(run_conv2d(r, a, nullptr, false, h->f_enc_conv0, &x));
    FCB_TRY(release2(r, a));
    for (size_t i = 0; i < h->f_enc_rb.size(); ++i) {
        Act2 sc, blk, d;
        FCB_TRY(run_resblock2d(r, x, h->f_enc_rb[i], &sc, &blk));
        FCB_TRY(release2(r, x));
        FCB_TRY(run_conv2d(r, sc, &blk, true, h->f_enc_down[i], &d));
        FCB_TRY(release2(r, sc));
        FCB_TRY(release2(r, blk));
        x = d;
    }
    if (x.F != 1) return fail(h, FCB_E_INVALID, "FreqCodec encoder: frequency axis did not reduce to 1 (check ratios / n_fft)");
    FCB_TRY(phase_end(r));
    // squeeze (ReshapeModule, seanet_encoder.py:326): [B][1][T][C] is already a 1-D channels-last tensor
    Act y1;
    y1.p = x.p; y1.T = x.T; y1.C = x.C; y1.clip_stride = (long long)x.T * x.C; y1.stats = x.stats; y1.coef = x.coef;
    y1.gamma = x.gamma; y1.beta = x.beta; y1.owned = true;
    FCB_TRY(phase_begin(r, FCB_PHASE_ENCODER_LSTM));
    if (c.lstm_layers > 0) {
        Act y;
        FCB_TRY(run_lstm(r, y1, h->enc_lstm, &y));
        FCB_TRY(release(r, y1));
        y1 = y;
    }
    Act f;
    FCB_TRY(run_conv(r, y1, nullptr, true, nullptr, h->enc_final, true, &f));
    FCB_TRY(release(r, y1));
    FCB_TRY(phase_end(r));
    *out = f;
    return FCB_OK;
}

// SEANetDecoder2d.forward + FreqCodec._decode_frame (mag_phase) + iSTFT + trim.
int run_decoder_freq(Run& r, const float* emb, int n_frames, const float* scale, float* wav_out, int out_len) {
    fcb_handle* h = r.h;
    const fcb_config& c = h->cfg;
    if (out_len <= 0 || out_len > fcb_decoded_length(h, n_frames))
        return fail(h, FCB_E_INVALID, "out_len must be in (0, fcb_decoded_length]");
    Act e;
    e.p = const_cast<float*>(emb); e.T = n_frames; e.C = c.dimension; e.clip_stride = (long long)n_frames * e.C;
    FCB_TRY(phase_begin(r, FCB_PHASE_DECODER_LSTM));
    Act a;
    FCB_TRY(run_conv(r, e, nullptr, false, nullptr, h->dec_conv0, true, &a));
    if (c.lstm_layers > 0) {
        Act y;
        FCB_TRY(run_lstm(r, a, h->dec_lstm, &y));
        FCB_TRY(release(r, a));
        a = y;
    }
    FCB_TRY(phase_end(r));
    FCB_TRY(phase_begin(r, FCB_PHASE_DECODER_CONV));
    // unsqueeze (seanet_decoder.py:235-241)
    Act2 sc, blk;
    sc.p = a.p; sc.F_raw = sc.F = 1; sc.T_raw = sc.T = a.T; sc.C = a.C; sc.stats = a.stats; sc.coef = a.coef;
    sc.gamma = a.gamma; sc.beta = a.beta; sc.owned = true;
    bool have_blk = false;
    for (size_t i = 0; i < h->f_dec_up.size(); ++i) {
        Act2 u;
        FCB_TRY(run_conv2d(r, sc, have_blk ? &blk : nullptr, true, h->f_dec_up[i], &u));
        FCB_TRY(release2(r, sc));
        if (have_blk) FCB_TRY(release2(r, blk));
        FCB_TRY(run_resblock2d(r, u, h->f_dec_rb[i], &sc, &blk));
        FCB_TRY(release2(r, u));
        have_blk = true;
    }
    Act2 f;
    FCB_TRY(run_conv2d(r, sc, have_blk ? &blk : nullptr, true, h->f_dec_final, &f));
    FCB_TRY(release2(r, sc));
    if (have_blk) FCB_TRY(release2(r, blk));
    const int n_bins = c.n_fft / 2 + 1;
    if (f.F != n_bins || f.C != 3) return fail(h, FCB_E_INVALID, "FreqCodec decoder: output is not [n_fft/2+1 bins x 3 channels]");
    float* frames = nullptr;
    FCB_TRY(alloc_f(r, &frames, (size_t)r.B * f.T * c.n_fft));
    if (h->stft_tc && !h->stft_packed) { h->stft_packed = true; FCB_TRY(pack_stft_bases(h)); }
    if (h->stft_tc && h->istft_w.n_tile > 0) {      // softplus(mag)*(re, im) rows -> inverse-DFT GEMM -> overlap-add
        float* Y = nullptr;
        FCB_TRY(alloc_f(r, &Y, (size_t)r.B * f.T * h->istft_ld));
        FCB_CK(launch_spec_rows(f.p, f.coef, r.B, f.F_raw, f.T_raw, n_bins, f.T, h->istft_ld, Y, r.st));
        FCB_TRY(run_plain_tc(r, Y, f.T, h->istft_w, f.T, frames));
        FCB_CK(launch_istft_ola(frames, scale, r.B, c.n_fft, c.stft_hop, f.T, out_len, wav_out, r.st));
        h->launches += 3;
        FCB_TRY(pool_free(r, Y));
    } else {
        FCB_CK(launch_istft(f.p, f.coef, r.B, f.F_raw, f.T_raw, c.n_fft, c.stft_hop, f.T, scale, frames, wav_out, out_len, r.st));
        h->launches += 2;
    }
    FCB_TRY(pool_free(r, frames));
    FCB_TRY(release2(r, f));
    FCB_TRY(phase_end(r));
    return FCB_OK;
}

// "stft_tc" (default): the windowed DFT / inverse-DFT bases as tensor-core conv weight images.
//  STFT : rows of 32 samples are the channels-last input, X[m][co] = sum_{k, ci} x[(m*s + k)*32 + ci] * Wf[k][ci][co] with
//         Wf = hann[n] cos(2 pi co n / N) for co < n_bins, -hann[n] sin(2 pi (co - n_bins) n / N) for the next n_bins columns;
//  iSTFT: frames[m][j] = sum_ci Y[m][ci] * Wi[ci][j], Wi = c_k cos(2 pi k j / N) hann[j] / N (ci = k), -c_k sin(.) hann[j] / N
//         (ci = n_bins + k), c_0 = c_{N/2} = 1 (their imaginary parts are ignored, as irfft does), c_k = 2 otherwise.
int pack_stft_bases(fcb_handle* h) {
    const fcb_config& c = h->cfg;
    const int N = c.n_fft, hop = c.stft_hop, n_bins = N / 2 + 1;
    h->stft_w.n_tile = 0; h->istft_w.n_tile = 0;
    if (!h->use_tc || N % 32 != 0 || hop % 32 != 0 || N < hop) return FCB_OK;
    const double two_pi = 6.283185307179586476925286766559;
    std::vector<double> hann(N);
    for (int n = 0; n < N; ++n) hann[n] = 0.5 - 0.5 * cos(two_pi * n / N);
    {   // forward
        const int K = N / 32, cout = (2 * n_bins + 127) / 128 * 128;
        if (!conv_tc_supported(32, cout, K, hop / 32, 1)) return FCB_OK;
        std::vector<float> wp((size_t)K * 32 * cout, 0.f), bias(cout, 0.f);
        for (int n = 0; n < N; ++n)
            for (int k = 0; k < n_bins; ++k) {
                const double ang = two_pi * (double)(((long long)k * n) % N) / N;
                wp[(size_t)n * cout + k] = (float)(hann[n] * cos(ang));
                wp[(size_t)n * cout + n_bins + k] = (float)(-hann[n] * sin(ang));
            }
        ConvW& o = h->stft_w;
        o.cin = 32; o.cout = cout; o.k = K; o.s = hop / 32;
        std::vector<float> img;
        const int n_tile = conv_tc_n_tile(cout);
        build_tc_image_f16(wp, K, 32, cout, n_tile, &img, &o.tc_scale);
        FCB_TRY(upload(h, img, &o.w_tc));
        FCB_TRY(upload(h, bias, &o.bias));
        o.n_tile = n_tile;
        h->stft_ld = cout;
    }
    {   // inverse
        const int cin = (2 * n_bins + 31) / 32 * 32, cout = N;
        if (!conv_tc_supported(cin, cout, 1, 1, 1)) return FCB_OK;
        std::vector<float> wp((size_t)cin * cout, 0.f), bias(cout, 0.f);
        for (int k = 0; k < n_bins; ++k) {
            const bool edge = (k == 0 || k == N / 2);
            for (int j = 0; j < N; ++j) {
                const double ang = two_pi * (double)(((long long)k * j) % N) / N;
                wp[(size_t)k * cout + j] = (float)((edge ? 1.0 : 2.0) * cos(ang) * hann[j] / N);
                wp[(size_t)(n_bins + k) * cout + j] = edge ? 0.f : (float)(-2.0 * sin(ang) * hann[j] / N);
            }
        }
        ConvW& o = h->istft_w;
        o.cin = cin; o.cout = cout; o.k = 1; o.s = 1;
        std::vector<float> img;
        const int n_tile = conv_tc_n_tile(cout);
        build_tc_image_f16(wp, 1, cin, cout, n_tile, &img, &o.tc_scale);
        FCB_TRY(upload(h, img, &o.w_tc));
        FCB_TRY(upload(h, bias, &o.bias));
        o.n_tile = n_tile;
        h->istft_ld = cin;
    }
    return FCB_OK;
}

// one plain tensor-core conv without padding, normalisation or statistics: out[B][T_out][cout] (used by the GEMM STFT / iSTFT)
int run_plain_tc(Run& r, const float* x, int T_in, const ConvW& L, int T_out, float* out) {
    fcb_handle* h = r.h;
    ConvParams p{};
    p.in0.x = x; p.in0.clip_stride = (long long)T_in * L.cin;
    p.T_in = T_in; p.C_in = L.cin; p.K = L.k; p.S = L.s; p.D = 1; p.pad_l = 0; p.T_ext = T_in; p.pad_zero = 1;
    p.w_tc = L.w_tc; p.n_tile = L.n_tile; p.tc_w_scale = L.tc_scale; p.bias = L.bias;
    p.out = out; p.T_out = T_out; p.C_out = L.cout; p.out_clip_stride = (long long)T_out * L.cout;
    int np = 0;
    FCB_CK(launch_conv_tc(p, r.B, r.st, &np));
    h->launches++;
    return FCB_OK;
}

int finalize_freq(fcb_handle* h) {
    const fcb_config& c = h->cfg;
    const int nf = c.n_filters, D = c.dimension, nr = c.n_ratios;
    FCB_TRY(pack_conv2d(h, "encoder.model.0", 3, nf, c.kernel_size, c.kernel_size, 1, 1, &h->f_enc_conv0, 4));
    int n = 1, mult = 1;
    for (int i = nr - 1; i >= 0; --i) {               // encoder applies the ratios reversed (seanet_encoder.py:288)
        const int fr = c.ratios_f[i], tr = c.ratios[i];
        ResBlock2W rb; Conv2W down;
        FCB_TRY(pack_resblock2d(h, "encoder.model." + std::to_string(n), mult * nf, &rb));
        FCB_TRY(pack_conv2d(h, "encoder.model." + std::to_string(n + 2), mult * nf, 2 * mult * nf, 2 * fr, 2 * tr, fr, tr, &down, 0,
                            conv_groups_of(mult * nf, c.conv_group_ratio)));
        h->f_enc_rb.push_back(rb); h->f_enc_down.push_back(down);
        mult *= 2; n += 3;
    }
    n += 1;                                             // ReshapeModule
    if (c.lstm_layers > 0) {
        FCB_TRY(pack_lstm(h, "encoder.model." + std::to_string(n), mult * nf, c.lstm_layers, &h->enc_lstm));
        n += 1;
    }
    FCB_TRY(pack_conv(h, "encoder.model." + std::to_string(n + 1), mult * nf, D, c.last_kernel_size, 1, &h->enc_final));
    FCB_TRY(pack_conv(h, "decoder.model.0", D, mult * nf, c.kernel_size, 1, &h->dec_conv0));
    n = 1;
    if (c.lstm_layers > 0) {
        FCB_TRY(pack_lstm(h, "decoder.model.1", mult * nf, c.lstm_layers, &h->dec_lstm));
        n = 2;
    }
    n += 1;                                             // ReshapeModule
    for (int i = 0; i < nr; ++i) {
        const int fr = c.ratios_f[i], tr = c.ratios[i];
        Conv2W up; ResBlock2W rb;
        FCB_TRY(pack_convtr2d(h, "decoder.model." + std::to_string(n + 1), mult * nf, mult * nf / 2, fr, tr, &up,
                              conv_groups_of(mult * nf, c.tr_conv_group_ratio)));
        FCB_TRY(pack_resblock2d(h, "decoder.model." + std::to_string(n + 2), mult * nf / 2, &rb));
        if (i == nr - 1) up.out_pad[0][1] = 1;         // SEANetDecoder2d last_out_padding default [(0, 1), (0, 0)]
        h->f_dec_up.push_back(up); h->f_dec_rb.push_back(rb);
        mult /= 2; n += 3;
    }
    FCB_TRY(pack_conv2d(h, "decoder.model." + std::to_string(n + 1), nf, 3, c.last_kernel_size, c.last_kernel_size, 1, 1, &h->f_dec_final));
    return FCB_OK;
}

int run_decoder(Run& r, const float* emb, int n_frames, const float* scale, float* wav_out, int out_len) {
    return r.h->cfg.arch == 1 ? run_decoder_freq(r, emb, n_frames, scale, wav_out, out_len)
                              : run_decoder_time(r, emb, n_frames, scale, wav_out, out_len);
}

int check_ready(fcb_handle* h) {
    if (!h) return FCB_E_INVALID;
    if (!h->finalized) return fail(h, FCB_E_STATE, "fcb_finalize has not been called");
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != h->device)
        return fail(h, FCB_E_STATE, "handle used on a different CUDA device than it was created on");
    return FCB_OK;
}

int do_encode(fcb_handle* h, const float* wav, int B, int L, int n_q, int64_t* codes, float* quant, float* scale,
              float* sub_quants, float* encoder_out, cudaStream_t st) {
    if (!wav || !codes || B <= 0 || L <= 0) return fail(h, FCB_E_INVALID, "fcb_encode: bad arguments");
    if (n_q <= 0 || n_q > h->cfg.num_quantizers) return fail(h, FCB_E_INVALID, "fcb_encode: n_q out of range");
    if (B > 512) return fail(h, FCB_E_INVALID, "fcb_encode: at most 512 clips per call (split the batch)");
    Run r{h, B, st};
    Act f;
    if (h->cfg.arch == 1) FCB_TRY(run_encoder_freq(r, wav, L, scale, &f));
    else FCB_TRY(run_encoder(r, wav, L, scale, &f));
    FCB_TRY(phase_begin(r, FCB_PHASE_RVQ));
    RvqParams q{};
    q.in = view_of(f);
    q.embed = h->embed; q.cnorm = h->cnorm;
    q.B = B; q.T = f.T; q.D = h->cfg.dimension; q.K = h->cfg.codebook_size; q.n_q = n_q;
    q.codes = reinterpret_cast<long long*>(codes);
    q.sub_quants = sub_quants; q.enc_out = encoder_out;
    q.embed_tc = h->embed_tc;
    q.allow_sliced = h->rvq_sliced;
    if (h->use_tc && h->embed_tc) {
        q.quant = nullptr;
        FCB_CK(launch_rvq_tc(q, st));
        h->launches++;
        if (quant) {   // quantized_out = ((0 + q_0) + q_1) + ... rebuilt from the codes (ddp_core_vq.py:408 order)
            FCB_CK(launch_embed_sum(q.codes, 1, h->embed, B, f.T, n_q, h->cfg.codebook_size, h->cfg.dimension, quant,
                                    h->err_flag, st));
            h->launches++;
        }
    } else {
        q.quant = quant;
        FCB_CK(launch_rvq(q, st));
        h->launches++;
    }
    FCB_TRY(release(r, f));
    FCB_TRY(phase_end(r));
    return FCB_OK;
}

}  // namespace

// =============================================================================================== C ABI
extern "C" {

const char* fcb_version(void) { return "funcodec_b200 0.1.0 sm_100a"; }

int fcb_create(const fcb_config* cfg, fcb_handle** out) {
    if (!cfg || !out) return FCB_E_INVALID;
    if (cfg->n_ratios < 1 || cfg->n_ratios > FCB_MAX_RATIOS || cfg->n_filters < 2 || cfg->dimension < 4 ||
        cfg->dimension % 4 != 0 || cfg->codebook_size < 1 || cfg->num_quantizers < 1 || cfg->lstm_layers < 0 ||
        cfg->kernel_size < 1 || cfg->last_kernel_size < 1 || cfg->residual_kernel_size < 1)
        return FCB_E_INVALID;
    for (int i = 0; i < cfg->n_ratios; ++i)
        if (cfg->ratios[i] < 1) return FCB_E_INVALID;
    if (cfg->arch != 0 && cfg->arch != 1) return FCB_E_INVALID;
    if (cfg->norm < 0 || cfg->norm > 2 || (cfg->causal != 0 && cfg->causal != 1)) return FCB_E_INVALID;
    if (cfg->causal && cfg->norm == 0) return FCB_E_INVALID;      // "GroupNorm doesn't support causal evaluation" (conv.py:46-47)
    if (cfg->arch == 1 && (cfg->norm != 0 || cfg->causal)) return FCB_E_INVALID;   // FreqCodec: time_group_norm, non-causal only
    if (cfg->channels < 0 || cfg->channels > 2) return FCB_E_INVALID;              // the reference asserts 0 < channels <= 2
    if (cfg->arch == 1 && cfg->channels == 2) return FCB_E_INVALID;                // FreqCodec STFTs x.squeeze(1): mono only
    if (cfg->arch == 1) {
        if (cfg->n_fft < 16 || cfg->n_fft % 2 != 0 || cfg->stft_hop < 1 || cfg->stft_hop > cfg->n_fft) return FCB_E_INVALID;
        for (int i = 0; i < cfg->n_ratios; ++i)
            if (cfg->ratios_f[i] < 1) return FCB_E_INVALID;
    }
    fcb_handle* h = new (std::nothrow) fcb_handle();
    if (!h) return FCB_E_NOMEM;
    h->cfg = *cfg;
    { const char* e = getenv("FCB_DISABLE_TC"); if (e && e[0] == '1') h->use_tc = false; }
    { const char* e = getenv("FCB_CONV2D_SMALL_COUT"); if (e && (e[0] == '0' || e[0] == '1')) h->conv2d_small_cout = e[0] - '0'; }
    { const char* e = getenv("FCB_STFT_TC"); if (e && (e[0] == '0' || e[0] == '1')) h->stft_tc = e[0] - '0'; }
    { const char* e = getenv("FCB_USE_TC2D"); if (e && e[0] >= '0' && e[0] <= '7' && !e[1]) h->use_tc2d = e[0] - '0'; }
    if (cudaGetDevice(&h->device) != cudaSuccess) { delete h; return FCB_E_CUDA; }
    // keep freed temporaries cached in the stream-ordered pool (no give-back between calls)
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, h->device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    *out = h;
    return FCB_OK;
}

int fcb_set_tensor(fcb_handle* h, const char* name, const float* data, int32_t ndim, const int64_t* shape) {
    if (!h || !name || !data || ndim < 0 || ndim > 4) return FCB_E_INVALID;
    if (h->finalized) return fail(h, FCB_E_STATE, "fcb_set_tensor after fcb_finalize");
    std::string n(name);
    // codebooks: stacked buffer of DistributedResidualVectorQuantization (use_ddp: true, ddp_core_vq.py:349-352) or the
    // per-layer buffers of ResidualVectorQuantization (use_ddp: false, core_vq.py:147-150) -- assembled in fcb_finalize
    const bool per_layer_embed = n.rfind("quantizer.rq.model.layers.", 0) == 0 && n.size() > 16 &&
                                 n.compare(n.size() - 16, 16, "._codebook.embed") == 0;
    const bool known = n.rfind("encoder.model.", 0) == 0 || n.rfind("decoder.model.", 0) == 0 ||
                       n == "quantizer.rq.model.embed" || per_layer_embed;
    if (!known) return 1;   // ignored (discriminator, EMA buffers, ...), like filter_state_dict
    HostTensor t;
    size_t cnt = 1;
    for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); cnt *= (size_t)shape[i]; }
    t.data.assign(data, data + cnt);
    h->host[n] = std::move(t);
    return FCB_OK;
}

int fcb_finalize(fcb_handle* h) {
    if (!h) return FCB_E_INVALID;
    if (h->finalized) return fail(h, FCB_E_STATE, "already finalized");
    const fcb_config& c = h->cfg;
    const int nf = c.n_filters, D = c.dimension;
    if (c.arch == 1) {
        FCB_TRY(finalize_freq(h));
    } else {
    const int ch = h->channels();
    FCB_TRY(pack_conv(h, "encoder.model.0", ch, nf, c.kernel_size, 1, &h->enc_conv0));
    int n = 1, mult = 1;
    const int nres = c.n_residual_layers > 0 ? c.n_residual_layers : 1, dbase = c.dilation_base > 0 ? c.dilation_base : 2;
    for (int i = c.n_ratios - 1; i >= 0; --i) {      // encoder applies the ratios reversed (seanet_encoder.py:102)
        const int ratio = c.ratios[i];
        ConvW down;
        int dil = 1;
        for (int j = 0; j < nres; ++j, dil *= dbase) {            // dilations dilation_base^j (seanet_encoder.py:122-128)
            ResBlockW rb;
            FCB_TRY(pack_resblock(h, "encoder.model." + std::to_string(n + j), mult * nf, &rb, dil));
            h->enc_rb.push_back(rb);
        }
        FCB_TRY(pack_conv(h, "encoder.model." + std::to_string(n + nres + 1), mult * nf, 2 * mult * nf, 2 * ratio, ratio, &down));
        h->enc_down.push_back(down);
        mult *= 2; n += nres + 2;
    }
    if (c.lstm_layers > 0) {
        FCB_TRY(pack_lstm(h, "encoder.model." + std::to_string(n), mult * nf, c.lstm_layers, &h->enc_lstm));
        n += 1;
    }
    FCB_TRY(pack_conv(h, "encoder.model." + std::to_string(n + 1), mult * nf, D, c.last_kernel_size, 1, &h->enc_final));

    FCB_TRY(pack_conv(h, "decoder.model.0", D, mult * nf, c.kernel_size, 1, &h->dec_conv0));
    n = 1;
    if (c.lstm_layers > 0) {
        FCB_TRY(pack_lstm(h, "decoder.model.1", mult * nf, c.lstm_layers, &h->dec_lstm));
        n = 2;
    }
    for (int i = 0; i < c.n_ratios; ++i) {
        const int ratio = c.ratios[i];
        ConvW up;
        FCB_TRY(pack_convtr(h, "decoder.model." + std::to_string(n + 1), mult * nf, mult * nf / 2, ratio, &up));
        h->dec_up.push_back(up);
        int dil = 1;
        for (int j = 0; j < nres; ++j, dil *= dbase) {
            ResBlockW rb;
            FCB_TRY(pack_resblock(h, "decoder.model." + std::to_string(n + 2 + j), mult * nf / 2, &rb, dil));
            h->dec_rb.push_back(rb);
        }
        mult /= 2; n += nres + 2;
    }
    FCB_TRY(pack_conv(h, "decoder.model." + std::to_string(n + 1), nf, ch, c.last_kernel_size, 1, &h->dec_final));
    // the stereo layers need the SIMT kernels: the first conv reads the planar waveform, and the decoder output goes
    // channels-last [T][2] into final_output_kernel; neither has a tensor-core form
    if (ch > 1 && (h->enc_conv0.n_tile > 0 || h->dec_final.n_tile > 0))
        return fail(h, FCB_E_INVALID, "stereo: the first encoder conv and the last decoder conv have no tensor-core path "
                    "for 2 channels (planar input / C_out = 2)");
    }

    if (!find(h, "quantizer.rq.model.embed") && find(h, "quantizer.rq.model.layers.0._codebook.embed")) {
        // use_ddp: false checkpoints (core_vq.py:147-150): one [K][D] buffer per stage, same semantics as the stacked tensor
        HostTensor st;
        st.shape = {c.num_quantizers, c.codebook_size, D};
        for (int q = 0; q < c.num_quantizers; ++q) {
            const HostTensor* e;
            FCB_TRY(need(h, "quantizer.rq.model.layers." + std::to_string(q) + "._codebook.embed", {c.codebook_size, D}, &e));
            st.data.insert(st.data.end(), e->data.begin(), e->data.end());
        }
        h->host["quantizer.rq.model.embed"] = std::move(st);
    }
    const HostTensor* emb;
    FCB_TRY(need(h, "quantizer.rq.model.embed", {c.num_quantizers, c.codebook_size, D}, &emb));
    if (const char* v = getenv("FCB_RVQ_SLICED")) h->rvq_sliced = atoi(v) != 0;
    {
        const int ds = rvq_simt_slice(D);
        if (ds == 0) return fail(h, FCB_E_INVALID, "dimension " + std::to_string(D) + " is too wide for the RVQ kernels");
        if (ds != D && !h->rvq_sliced)
            return fail(h, FCB_E_INVALID, "dimension " + std::to_string(D) + ": the RVQ kernels keep the residual, the running sum and a "
                        "128-codeword chunk in shared memory, which fits D <= 260; the column-sliced kernel for wider embeddings is "
                        "switched off (fcb_set_option(\"rvq_sliced\", 0) / FCB_RVQ_SLICED=0)");
    }
    FCB_TRY(upload(h, emb->data, &h->embed));
    if (h->use_tc && rvq_tc_supported(D, c.codebook_size)) {
        // per stage: [1][D][K] "weights" (codeword = output channel) -> slab images, stages concatenated
        std::vector<float> all, wp((size_t)D * c.codebook_size), img;
        for (int q = 0; q < c.num_quantizers; ++q) {
            const float* e = emb->data.data() + (size_t)q * c.codebook_size * D;
            for (int k = 0; k < c.codebook_size; ++k)
                for (int d = 0; d < D; ++d) wp[(size_t)d * c.codebook_size + k] = e[(size_t)k * D + d];
            build_tc_image_tf32(wp, 1, D, c.codebook_size, RVQ_TC_N, &img);
            all.insert(all.end(), img.begin(), img.end());
        }
        FCB_TRY(upload(h, all, &h->embed_tc));
    }
    FCB_CK(cudaMalloc((void**)&h->cnorm, (size_t)c.num_quantizers * c.codebook_size * sizeof(float)));
    h->dev_allocs.push_back(h->cnorm);
    FCB_CK(cudaMalloc((void**)&h->err_flag, sizeof(int)));
    h->dev_allocs.push_back(h->err_flag);
    FCB_CK(cudaMemset(h->err_flag, 0, sizeof(int)));
    FCB_CK(cudaMalloc((void**)&h->lstm_barrier, 64 * sizeof(unsigned)));
    h->dev_allocs.push_back(h->lstm_barrier);
    if (getenv("FCB_LSTM_TRACE")) {
        FCB_CK(cudaMallocManaged((void**)&h->lstm_trace, LSTM_TRACE_ITEMS * 8 * sizeof(unsigned long long)));
        FCB_CK(cudaMemset(h->lstm_trace, 0, LSTM_TRACE_ITEMS * 8 * sizeof(unsigned long long)));
        h->dev_allocs.push_back(h->lstm_trace);
    }
    FCB_CK(launch_code_norms(h->embed, h->cnorm, c.num_quantizers * c.codebook_size, D, 0));
    h->launches++;
    FCB_CK(cudaDeviceSynchronize());
    h->host.clear();
    if (h->cfg.arch == 0) {   // name map for fcb_debug_conv1d (vectors are final now: pointers stay valid)
        const fcb_config& cc = h->cfg;
        h->by_name["encoder.model.0"] = &h->enc_conv0;
        int nn = 1;
        const int nres = cc.n_residual_layers > 0 ? cc.n_residual_layers : 1;
        for (size_t i = 0; i < h->enc_down.size(); ++i, nn += nres + 2) {
            for (int j = 0; j < nres; ++j) {
                const std::string pre = "encoder.model." + std::to_string(nn + j);
                h->by_name[pre + ".block.1"] = &h->enc_rb[i * nres + j].c1;
                h->by_name[pre + ".block.3"] = &h->enc_rb[i * nres + j].c2;
                h->by_name[pre + ".shortcut"] = &h->enc_rb[i * nres + j].sc;
            }
            h->by_name["encoder.model." + std::to_string(nn + nres + 1)] = &h->enc_down[i];
        }
        if (cc.lstm_layers > 0) {
            for (int l = 0; l < cc.lstm_layers; ++l) h->by_name["encoder.model." + std::to_string(nn) + ".lstm.ih" + std::to_string(l)] = &h->enc_lstm.ih[l];
            nn += 1;
        }
        h->by_name["encoder.model." + std::to_string(nn + 1)] = &h->enc_final;
        h->by_name["decoder.model.0"] = &h->dec_conv0;
        nn = cc.lstm_layers > 0 ? 2 : 1;
        for (size_t i = 0; i < h->dec_up.size(); ++i, nn += nres + 2) {
            h->by_name["decoder.model." + std::to_string(nn + 1)] = &h->dec_up[i];
            for (int j = 0; j < nres; ++j) {
                const std::string pre = "decoder.model." + std::to_string(nn + 2 + j);
                h->by_name[pre + ".block.1"] = &h->dec_rb[i * nres + j].c1;
                h->by_name[pre + ".block.3"] = &h->dec_rb[i * nres + j].c2;
                h->by_name[pre + ".shortcut"] = &h->dec_rb[i * nres + j].sc;
            }
        }
        h->by_name["decoder.model." + std::to_string(nn + 1)] = &h->dec_final;
    }
    if (h->cfg.arch == 1) {   // name map for fcb_debug_conv2d
        const fcb_config& cc = h->cfg;
        h->by_name2["encoder.model.0"] = &h->f_enc_conv0;
        int nn = 1;
        for (size_t i = 0; i < h->f_enc_rb.size(); ++i, nn += 3) {
            const std::string pre = "encoder.model." + std::to_string(nn);
            h->by_name2[pre + ".block.1"] = &h->f_enc_rb[i].c1;
            h->by_name2[pre + ".block.3"] = &h->f_enc_rb[i].c2;
            h->by_name2[pre + ".shortcut"] = &h->f_enc_rb[i].sc;
            h->by_name2["encoder.model." + std::to_string(nn + 2)] = &h->f_enc_down[i];
        }
        nn = (cc.lstm_layers > 0 ? 2 : 1) + 1;          // decoder: conv0, [lstm], ReshapeModule
        for (size_t i = 0; i < h->f_dec_up.size(); ++i, nn += 3) {
            h->by_name2["decoder.model." + std::to_string(nn + 1)] = &h->f_dec_up[i];
            const std::string pre = "decoder.model." + std::to_string(nn + 2);
            h->by_name2[pre + ".block.1"] = &h->f_dec_rb[i].c1;
            h->by_name2[pre + ".block.3"] = &h->f_dec_rb[i].c2;
            h->by_name2[pre + ".shortcut"] = &h->f_dec_rb[i].sc;
        }
        h->by_name2["decoder.model." + std::to_string(nn + 1)] = &h->f_dec_final;
    }
    h->finalized = true;
    return FCB_OK;
}

int fcb_num_frames(const fcb_handle* h, int32_t L) {
    if (!h || L <= 0) return FCB_E_INVALID;
    if (h->cfg.arch == 1) {          // STFT frames (center=True): 1 + L / hop, then the encoder's time strides
        const int ts = 1 + L / h->cfg.stft_hop, tp = h->tprod();
        return (ts + tp - 1) / tp;
    }
    const int hop = h->hop();
    return (L + hop - 1) / hop;
}

int fcb_decoded_length(const fcb_handle* h, int32_t n_frames) {
    if (!h || n_frames <= 0) return FCB_E_INVALID;
    if (h->cfg.arch == 1) return h->cfg.stft_hop * (n_frames * h->tprod() - 1);   // torch.istft(center=True, length=None)
    return n_frames * h->hop();
}

int fcb_num_quantizers_for_bandwidth(const fcb_handle* h, double bandwidth) {
    if (!h) return FCB_E_INVALID;
    const double bw_per_q = log2((double)h->cfg.codebook_size) * h->cfg.sample_rate / h->hop();
    int n_q = h->cfg.num_quantizers;
    if (bandwidth > 0.0) {
        n_q = (int)floor(bandwidth / bw_per_q);
        if (n_q < 1) n_q = 1;
    }
    return n_q;
}

int fcb_encode(fcb_handle* h, const float* wav, int32_t B, int32_t L, int32_t n_q, int64_t* codes, float* quant,
               float* scale, float* sub_quants, float* encoder_out, void* stream) {
    FCB_TRY(check_ready(h));
    return do_encode(h, wav, B, L, n_q, codes, quant, scale, sub_quants, encoder_out, (cudaStream_t)stream);
}

int fcb_decode_emb(fcb_handle* h, const float* emb, int32_t B, int32_t n_frames, const float* scale, float* wav_out,
                   int32_t out_len, void* stream) {
    FCB_TRY(check_ready(h));
    if (!emb || !wav_out || B <= 0 || n_frames <= 0) return fail(h, FCB_E_INVALID, "fcb_decode_emb: bad arguments");
    Run r{h, B, (cudaStream_t)stream};
    return run_decoder(r, emb, n_frames, scale, wav_out, out_len);
}

int fcb_decode_codes(fcb_handle* h, const int64_t* codes, int32_t B, int32_t n_frames, int32_t n_q, float* emb_out,
                     float* wav_out, int32_t out_len, void* stream) {
    FCB_TRY(check_ready(h));
    if (!codes || !wav_out || B <= 0 || n_frames <= 0) return fail(h, FCB_E_INVALID, "fcb_decode_codes: bad arguments");
    if (n_q <= 0 || n_q > h->cfg.num_quantizers) return fail(h, FCB_E_INVALID, "fcb_decode_codes: n_q out of range");
    cudaStream_t st = (cudaStream_t)stream;
    Run r{h, B, st};
    float* emb = emb_out;
    const size_t n = (size_t)B * n_frames * h->cfg.dimension;
    if (!emb) FCB_TRY(alloc_f(r, &emb, n));
    FCB_TRY(phase_begin(r, FCB_PHASE_RVQ));
    FCB_CK(launch_embed_sum(reinterpret_cast<const long long*>(codes), 0, h->embed, B, n_frames, n_q, h->cfg.codebook_size,
                            h->cfg.dimension, emb, h->err_flag, st));
    h->launches++;
    FCB_TRY(phase_end(r));
    int rc = run_decoder(r, emb, n_frames, nullptr, wav_out, out_len);
    if (!emb_out) FCB_TRY(pool_free(r, emb));
    return rc;
}

int fcb_roundtrip(fcb_handle* h, const float* wav, int32_t B, int32_t L, int32_t n_q, int32_t use_scale, int64_t* codes,
                  float* quant, float* scale, float* sub_quants, float* recon, void* stream) {
    FCB_TRY(check_ready(h));
    if (!recon) return fail(h, FCB_E_INVALID, "fcb_roundtrip: recon is required");
    cudaStream_t st = (cudaStream_t)stream;
    Run r{h, B, st};
    const int Tf = fcb_num_frames(h, L);
    const size_t nq = (size_t)B * Tf * h->cfg.dimension;
    float* q = quant;
    float* sc = scale;
    if (!q) FCB_TRY(alloc_f(r, &q, nq));
    if (!sc) FCB_TRY(alloc_f(r, &sc, B));
    int rc = do_encode(h, wav, B, L, n_q, codes, q, sc, sub_quants, nullptr, st);
    if (rc == FCB_OK) {
        const bool apply = use_scale && h->cfg.audio_normalize;
        rc = run_decoder(r, q, Tf, apply ? sc : nullptr, recon, L);
    }
    if (!quant) FCB_TRY(pool_free(r, q));
    if (!scale) FCB_TRY(pool_free(r, sc));
    return rc;
}

// Pure arithmetic (no device, no handle): error text through *why when not representable.
static int plan_segments_hop(int hop, int32_t L, int32_t seg_len, int32_t stride, fcb_segment_plan* plan, const char** why) {
    if (hop <= 0 || L <= 0 || seg_len <= 0 || stride <= 0 || stride > seg_len) {
        *why = "fcb_plan_segments: need hop > 0, L > 0 and 0 < stride <= seg_len";
        return FCB_E_INVALID;
    }
    fcb_segment_plan p{};
    p.n_seg = (L + stride - 1) / stride;                                    // len(range(0, L, stride))
    p.n_full = L >= seg_len ? (L - seg_len) / stride + 1 : 0;              // offsets with a whole segment left
    if (p.n_full > p.n_seg) p.n_full = p.n_seg;
    p.n_tail = p.n_seg - p.n_full;
    if (p.n_tail > FCB_MAX_TAIL_SEGMENTS) {
        *why = "fcb_plan_segments: too many short trailing segments (overlap too high)";
        return FCB_E_INVALID;
    }
    p.frames_full = (seg_len + hop - 1) / hop;
    p.decoded_full = p.frames_full * hop;
    p.total_frames = (int64_t)p.n_full * p.frames_full;
    for (int i = 0; i < p.n_tail; ++i) {
        p.tail_len[i] = L - (p.n_full + i) * stride;
        p.tail_frames[i] = (p.tail_len[i] + hop - 1) / hop;
        p.total_frames += p.tail_frames[i];
    }
    // _linear_overlap_add sizes its output from the LAST frame (codec_basic.py:101); an earlier frame that ends later raises
    const int dl_last = p.n_tail ? p.tail_frames[p.n_tail - 1] * hop : p.decoded_full;
    const long long total = (long long)stride * (p.n_seg - 1) + dl_last;
    for (int i = 0; i < p.n_seg; ++i) {
        const int dl = i < p.n_full ? p.decoded_full : p.tail_frames[i - p.n_full] * hop;
        if ((long long)i * stride + dl > total) {
            *why = "segment plan not representable: a decoded segment ends after the final one "
                   "(the reference's _linear_overlap_add raises here)";
            return FCB_E_INVALID;
        }
    }
    *plan = p;
    return FCB_OK;
}

int fcb_plan_segments_for_hop(int32_t hop, int32_t L, int32_t seg_len, int32_t stride, fcb_segment_plan* plan) {
    if (!plan) return FCB_E_INVALID;
    const char* why = "";
    return plan_segments_hop(hop, L, seg_len, stride, plan, &why);
}

int fcb_plan_segments(fcb_handle* h, int32_t L, int32_t seg_len, int32_t stride, fcb_segment_plan* plan) {
    if (!h || !plan) return FCB_E_INVALID;
    if (h->cfg.arch != 0) return fail(h, FCB_E_INVALID, "segmented processing supports the time-domain Encodec only");
    const char* why = "";
    const int rc = plan_segments_hop(h->hop(), L, seg_len, stride, plan, &why);
    if (rc != FCB_OK) return fail(h, rc, why);
    return FCB_OK;
}

int fcb_roundtrip_segmented(fcb_handle* h, const float* wav, int32_t B, int32_t L, int32_t seg_len, int32_t stride,
                            int32_t n_q, int32_t use_scale, int64_t* codes, float* quant, float* scale, float* recon,
                            void* stream) {
    FCB_TRY(check_ready(h));
    if (!wav || !codes || B <= 0) return fail(h, FCB_E_INVALID, "fcb_roundtrip_segmented: bad arguments");
    if (B > 512) return fail(h, FCB_E_INVALID, "fcb_roundtrip_segmented: at most 512 clips per call (split the batch)");
    fcb_segment_plan pl;
    FCB_TRY(fcb_plan_segments(h, L, seg_len, stride, &pl));
    cudaStream_t st = (cudaStream_t)stream;
    const int D = h->cfg.dimension, hop = h->hop();
    const int C = h->channels();           // a planar clip [C][L] is C rows for the gather and overlap-add kernels
    const bool apply = use_scale && h->cfg.audio_normalize;
    Run r{h, B, st};                       // owner of the temporaries that span the whole call
    OlaParams ola{};
    float* frames_full = nullptr;
    if (recon && pl.n_full > 0) FCB_TRY(alloc_f(r, &frames_full, (size_t)pl.n_full * B * C * pl.decoded_full));
    // ---- the full-length segments: one batch of n_full*B clips, in chunks of <= 512 clips
    const int n_clips = pl.n_full * B, T0 = pl.frames_full;
    for (int c0 = 0; c0 < n_clips; ) {
        // whole segments per chunk when possible (gather writes segment-major blocks)
        int segs = 512 / B;
        if (segs < 1) segs = 1;
        const int s0 = c0 / B;
        if (segs > pl.n_full - s0) segs = pl.n_full - s0;
        const int nc = segs * B;
        Run rc{h, nc, st};
        float* x = nullptr;
        FCB_TRY(alloc_f(rc, &x, (size_t)nc * C * seg_len));
        FCB_CK(launch_gather_segments(wav, B * C, L, seg_len, stride, s0, segs, x, st));
        h->launches++;
        float* q = quant ? quant + (size_t)c0 * T0 * D : nullptr;
        float* sc = scale ? scale + c0 : nullptr;
        if (!q) FCB_TRY(alloc_f(rc, &q, (size_t)nc * T0 * D));
        if (!sc) FCB_TRY(alloc_f(rc, &sc, nc));
        const bool whole = (nc == n_clips);
        int64_t* cdst = codes + (size_t)c0 * T0;                         // [n_q][n_clips][T0], this chunk's clips
        int64_t* ctmp = cdst;
        if (!whole) FCB_TRY(pool_alloc(rc, (void**)&ctmp, (size_t)n_q * nc * T0 * sizeof(int64_t)));
        FCB_TRY(do_encode(h, x, nc, seg_len, n_q, ctmp, q, sc, nullptr, nullptr, st));
        if (!whole)
            FCB_CK(cudaMemcpy2DAsync(cdst, (size_t)n_clips * T0 * sizeof(int64_t), ctmp, (size_t)nc * T0 * sizeof(int64_t),
                                     (size_t)nc * T0 * sizeof(int64_t), n_q, cudaMemcpyDeviceToDevice, st));
        if (recon) FCB_TRY(run_decoder(rc, q, T0, apply ? sc : nullptr, frames_full + (size_t)c0 * C * pl.decoded_full, pl.decoded_full));
        c0 += nc;
    }
    // ---- the shorter trailing segments, one by one
    size_t code_off = (size_t)n_q * n_clips * T0, quant_off = (size_t)n_clips * T0 * D;
    for (int i = 0; i < pl.n_tail; ++i) {
        const int len = pl.tail_len[i], Ti = pl.tail_frames[i], dl = Ti * hop;
        Run rc{h, B, st};
        float* x = nullptr;
        FCB_TRY(alloc_f(rc, &x, (size_t)B * C * len));
        FCB_CK(launch_gather_segments(wav, B * C, L, len, stride, pl.n_full + i, 1, x, st));
        h->launches++;
        float* q = quant ? quant + quant_off : nullptr;
        float* sc = scale ? scale + (size_t)(pl.n_full + i) * B : nullptr;
        if (!q) FCB_TRY(alloc_f(rc, &q, (size_t)B * Ti * D));
        if (!sc) FCB_TRY(alloc_f(rc, &sc, B));
        FCB_TRY(do_encode(h, x, B, len, n_q, codes + code_off, q, sc, nullptr, nullptr, st));
        if (recon) {
            float* fr = nullptr;
            FCB_TRY(alloc_f(r, &fr, (size_t)B * C * dl));
            FCB_TRY(run_decoder(rc, q, Ti, apply ? sc : nullptr, fr, dl));
            ola.tail[i] = fr; ola.tail_dl[i] = dl;
        }
        code_off += (size_t)n_q * B * Ti;
        quant_off += (size_t)B * Ti * D;
    }
    if (recon) {
        ola.full = frames_full; ola.n_seg = pl.n_seg; ola.n_full = pl.n_full;
        ola.dl0 = pl.n_full > 0 ? pl.decoded_full : ola.tail_dl[0];       // weights come from the FIRST frame's length
        ola.stride = stride; ola.B = B * C; ola.out_len = L; ola.out = recon;
        FCB_CK(launch_overlap_add(ola, st));
        h->launches++;
    }
    return FCB_OK;
}

int fcb_roundtrip_host(fcb_handle* h, const float* wav_host, int32_t B, int32_t L, int32_t n_q, int32_t use_scale,
                       int64_t* codes_host, float* recon_host, void* stream) {
    FCB_TRY(check_ready(h));
    if (!wav_host || !codes_host || !recon_host || B <= 0 || L <= 0)
        return fail(h, FCB_E_INVALID, "fcb_roundtrip_host: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    Run r{h, B, st};
    const int Tf = fcb_num_frames(h, L);
    const size_t n_wav = (size_t)B * h->channels() * L;
    float *d_wav, *d_recon;
    int64_t* d_codes;
    FCB_TRY(alloc_f(r, &d_wav, n_wav));
    FCB_TRY(alloc_f(r, &d_recon, n_wav));
    FCB_TRY(pool_alloc(r, (void**)&d_codes, (size_t)n_q * B * Tf * sizeof(int64_t)));
    FCB_CK(cudaMemcpyAsync(d_wav, wav_host, n_wav * sizeof(float), cudaMemcpyHostToDevice, st));
    int rc = fcb_roundtrip(h, d_wav, B, L, n_q, use_scale, d_codes, nullptr, nullptr, nullptr, d_recon, stream);
    if (rc == FCB_OK) {
        FCB_CK(cudaMemcpyAsync(codes_host, d_codes, (size_t)n_q * B * Tf * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        FCB_CK(cudaMemcpyAsync(recon_host, d_recon, n_wav * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    FCB_TRY(pool_free(r, d_wav));
    FCB_TRY(pool_free(r, d_recon));
    FCB_TRY(pool_free(r, d_codes));
    FCB_CK(cudaStreamSynchronize(st));
    return rc;
}

int fcb_check_errors(fcb_handle* h, void* stream) {
    FCB_TRY(check_ready(h));
    cudaStream_t st = (cudaStream_t)stream;
    int flag = 0;
    FCB_CK(cudaMemcpyAsync(&flag, h->err_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    FCB_CK(cudaStreamSynchronize(st));
    if (flag) {
        FCB_CK(cudaMemsetAsync(h->err_flag, 0, sizeof(int), st));
        return fail(h, FCB_E_INVALID, "token index out of range [0, codebook_size) in fcb_decode_codes (the reference's F.embedding raises here)");
    }
    return FCB_OK;
}

int64_t fcb_launch_count(const fcb_handle* h) { return h ? h->launches : -1; }

int fcb_set_option(fcb_handle* h, const char* key, int32_t value) {
    if (!h || !key) return FCB_E_INVALID;
    if (strcmp(key, "use_tc") == 0) {
        if (h->finalized && value && !h->use_tc) return fail(h, FCB_E_STATE, "use_tc can only be enabled before fcb_finalize");
        h->use_tc = value != 0;
        return FCB_OK;
    }
    if (strcmp(key, "stft_tc") == 0) {             // STFT / iSTFT as tensor-core GEMMs (default) vs the direct-DFT kernels
        h->stft_tc = value != 0;
        return FCB_OK;
    }
    if (strcmp(key, "rvq_sliced") == 0) {          // column-sliced fp32 RVQ kernel for D > 260 (default on; 0: refuse such a D)
        if (h->finalized) return fail(h, FCB_E_STATE, "rvq_sliced must be set before fcb_finalize");
        h->rvq_sliced = value != 0;
        return FCB_OK;
    }
    if (strcmp(key, "conv2d_small_cout") == 0) {   // halo-tile SIMT kernel (default) vs the padded tensor-core n-tile
        h->conv2d_small_cout = value != 0;
        return FCB_OK;
    }
    if (strcmp(key, "use_tc2d") == 0) {     // bit mask of 2-D layer classes on the tensor-core path (see Conv2W::tc_class)
        if (value < 0 || value > 7) return fail(h, FCB_E_INVALID, "use_tc2d must be a bit mask in [0, 7]");
        h->use_tc2d = value;
        return FCB_OK;
    }
    return fail(h, FCB_E_INVALID, std::string("unknown option: ") + key);
}

int fcb_debug_conv2d(fcb_handle* h, const char* layer, const float* x, int32_t B, int32_t F, int32_t T, int32_t elu,
                     float* y, int64_t y_capacity, float* stats, int32_t* dims, void* stream) {
    FCB_TRY(check_ready(h));
    if (!layer || !x || !y || !dims || B <= 0 || F <= 0 || T <= 0) return fail(h, FCB_E_INVALID, "fcb_debug_conv2d: bad arguments");
    std::string n(layer);
    auto it = h->by_name2.find(n);
    if (it == h->by_name2.end()) return fail(h, FCB_E_INVALID, "fcb_debug_conv2d: unknown layer " + n);
    const Conv2W* L = it->second;
    Run r{h, B, (cudaStream_t)stream};
    Act2 in;
    in.p = const_cast<float*>(x); in.F_raw = in.F = F; in.T_raw = in.T = T; in.C = L->cin;
    Act2 o;
    FCB_TRY(run_conv2d(r, in, nullptr, elu != 0, *L, &o));
    const long long total = (long long)B * o.F_raw * o.T_raw * o.C;
    if (total > y_capacity) { release2(r, o); return fail(h, FCB_E_INVALID, "fcb_debug_conv2d: y too small"); }
    FCB_CK(cudaMemcpyAsync(y, o.p, (size_t)total * sizeof(float), cudaMemcpyDeviceToDevice, r.st));
    if (stats) FCB_CK(cudaMemcpyAsync(stats, o.stats, (size_t)B * 2 * sizeof(float), cudaMemcpyDeviceToDevice, r.st));
    dims[0] = o.F_raw; dims[1] = o.T_raw; dims[2] = o.C; dims[3] = o.f_off; dims[4] = o.t_off; dims[5] = o.F; dims[6] = o.T;
    dims[7] = L->cin;
    FCB_TRY(release2(r, o));
    return FCB_OK;
}

int fcb_debug_conv1d(fcb_handle* h, const char* layer, const float* x, int32_t B, int32_t T, int32_t elu,
                     float* y, int64_t y_capacity, float* stats, int32_t* t_out, int32_t* c_out, int32_t* row_off,
                     void* stream) {
    FCB_TRY(check_ready(h));
    if (!layer || !x || !y || !t_out || !c_out || !row_off) return fail(h, FCB_E_INVALID, "fcb_debug_conv1d: bad arguments");
    const ConvW* L = nullptr;
    std::string n(layer);
    auto it = h->by_name.find(n);
    if (it == h->by_name.end()) return fail(h, FCB_E_INVALID, "fcb_debug_conv1d: unknown layer " + n);
    L = it->second;
    Run r{h, B, (cudaStream_t)stream};
    Act in;
    in.p = const_cast<float*>(x); in.T = T; in.C = L->cin; in.clip_stride = (long long)T * L->cin;
    if (L == &h->enc_conv0 && L->cin > 1) in.ch_stride = T;      // the stereo first conv reads the planar waveform layout
    Act o;
    FCB_TRY(run_conv(r, in, nullptr, elu != 0, nullptr, *L, stats != nullptr, &o));
    const long long rows = o.clip_stride / o.C;
    if ((long long)B * o.clip_stride > y_capacity) { release(r, o); return fail(h, FCB_E_INVALID, "fcb_debug_conv1d: y too small"); }
    FCB_CK(cudaMemcpyAsync(y, o.p, (size_t)B * o.clip_stride * sizeof(float), cudaMemcpyDeviceToDevice, r.st));
    if (stats) FCB_CK(cudaMemcpyAsync(stats, o.stats, (size_t)B * 2 * sizeof(float), cudaMemcpyDeviceToDevice, r.st));
    *t_out = (int32_t)rows; *c_out = o.C; *row_off = o.row_off;
    FCB_TRY(release(r, o));
    return FCB_OK;
}

int fcb_set_profiling(fcb_handle* h, int32_t enabled) {
    if (!h) return FCB_E_INVALID;
    if (enabled && !h->ev_created) {
        for (int i = 0; i < FCB_NUM_PHASES; ++i)
            for (int j = 0; j < 2; ++j) FCB_CK(cudaEventCreate(&h->ev[i][j]));
        h->ev_created = true;
    }
    h->profiling = enabled != 0;
    for (int i = 0; i < FCB_NUM_PHASES; ++i) h->ev_used[i] = false;
    return FCB_OK;
}

int fcb_get_phase_ms(fcb_handle* h, float* ms_out) {
    if (!h || !ms_out) return FCB_E_INVALID;
    for (int i = 0; i < FCB_NUM_PHASES; ++i) {
        ms_out[i] = 0.f;
        if (h->ev_created && h->ev_used[i]) {
            FCB_CK(cudaEventSynchronize(h->ev[i][1]));
            FCB_CK(cudaEventElapsedTime(&ms_out[i], h->ev[i][0], h->ev[i][1]));
        }
    }
    return FCB_OK;
}

const char* fcb_last_error(const fcb_handle* h) { return h ? h->err.c_str() : "null handle"; }

void fcb_destroy(fcb_handle* h) {
    if (!h) return;
    if (h->lstm_trace) {      // PROFILING ONLY: the last LSTM layer launch's per-item stamps of CTA 0 (ns, relative)
        cudaDeviceSynchronize();
        const unsigned long long* tr = h->lstm_trace;
        unsigned long long t0 = ~0ull;
        for (int i = 0; i < LSTM_TRACE_ITEMS * 8; ++i) if (tr[i] && tr[i] < t0) t0 = tr[i];
        fprintf(stderr, "LSTM trace (CTA 0, ns since first stamp): item | hs_empty poll_ok | h_in fma_done red_out | red_in published\n");
        for (int i = 0; i < LSTM_TRACE_ITEMS; ++i) {
            fprintf(stderr, "item %3d |", i);
            for (int e = 0; e < 7; ++e) fprintf(stderr, " %8lld", tr[i * 8 + e] ? (long long)(tr[i * 8 + e] - t0) : -1ll);
            fprintf(stderr, "\n");
        }
    }
    for (void* p : h->dev_allocs) cudaFree(p);
    if (h->ev_created)
        for (int i = 0; i < FCB_NUM_PHASES; ++i)
            for (int j = 0; j < 2; ++j) cudaEventDestroy(h->ev[i][j]);
    delete h;
}

}  // extern "C"
