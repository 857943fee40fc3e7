/*
 * funcodec_b200 -- C ABI of the B200-native (sm_100a) codec encode -> RVQ -> decode hot path.
 *
 * The reference (modelscope/FunCodec) is pure Python and has no FFI; the seam this library sits
 * under is the method seam of its `Encodec` model class (SURVEY.md section 8(b)):
 *     Encodec.inference / inference_encoding   funcodec/models/codec_basic.py:670-764
 *     Encodec.inference_decoding               funcodec/models/codec_basic.py:766-802
 *     Encodec.inference_decoding_emb           funcodec/models/codec_basic.py:804-836
 * as called by Speech2Token.__call__            funcodec/bin/codec_inference.py:86-134.
 * The reference-side binding is a ctypes stub (INTEGRATION.md); funcodec_b200/encodec.py is that stub.
 *
 * Conventions
 *   - plain C types only; no torch types.  All *device* pointers are caller-owned CUDA global memory on
 *     the device that was current at fcb_create(); `stream` is a cudaStream_t passed as void*.
 *   - every call is asynchronous on `stream` (no host synchronisation) unless stated otherwise.
 *   - return value: 0 = OK, negative = error (FCB_E_*); fcb_last_error() gives the text.  No C++
 *     exception crosses the ABI.  One handle per caller thread/stream; handles are not internally locked.
 *   - tensors use the reference's user-facing layouts: wav [B, L] fp32 ([B, 2, L] channel-planar for a stereo handle,
 *     fcb_config.channels = 2: every wav / wav_out / recon buffer below then holds 2 * L samples per clip); codes int64
 *     [n_q, B, T'] (encode side) and [B, T', n_q] (decode side, codec_basic.py:789); embeddings
 *     [B, T', D] fp32; sub_quants [n_q, B, D, T'] fp32.
 */
#ifndef FUNCODEC_B200_H_
#define FUNCODEC_B200_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define FCB_API __attribute__((visibility("default")))
#else
#define FCB_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define FCB_OK            0
#define FCB_E_INVALID    -1   /* bad argument / shape / name */
#define FCB_E_STATE      -2   /* call order (e.g. encode before finalize) */
#define FCB_E_CUDA       -3   /* CUDA runtime error */
#define FCB_E_MISSING    -4   /* a required tensor was never set */
#define FCB_E_NOMEM      -5

#define FCB_MAX_RATIOS 8

/* Hyper-parameters == the YAML keys GANSpeechCodecTask.build_model consumes
 * (funcodec/tasks/gan_speech_codec.py:301-358; egs/LibriTTS/codec/conf/encodec_16k_n32_600k_step*.yaml). */
typedef struct fcb_config {
    int32_t n_ratios;
    int32_t ratios[FCB_MAX_RATIOS]; /* decoder order, e.g. {8,5,4,2,2}; the encoder applies them reversed */
    int32_t n_filters;              /* 32 */
    int32_t dimension;              /* D = 128 */
    int32_t kernel_size;            /* 7 */
    int32_t last_kernel_size;       /* 7 */
    int32_t residual_kernel_size;   /* 3 */
    int32_t lstm_layers;            /* 2 (0 disables the SLSTM) */
    int32_t codebook_size;          /* K = 1024 */
    int32_t num_quantizers;         /* n_q max = 32 */
    int32_t sample_rate;            /* 16000 */
    int32_t audio_normalize;        /* model_conf.audio_normalize */
    float   gn_eps;                 /* nn.GroupNorm eps, 1e-5 */
    /* FreqCodec variant (funcodec/models/codec_freq.py, codec_domain ['mag_phase','mag_phase']): arch = 1.  ratios[] then
     * holds the TIME ratios and ratios_f[] the FREQUENCY ratios of encoder_conf.ratios [[f, t], ...]; in_channels = 3. */
    int32_t arch;                   /* 0: time-domain Encodec (codec_basic.py); 1: FreqCodec mag_phase (codec_freq.py) */
    int32_t ratios_f[FCB_MAX_RATIOS];
    int32_t n_fft;                  /* 512 */
    int32_t stft_hop;               /* 160 */
    /* grouped 2-D convs (arch 1): encoder_conf / decoder_conf conv_group_ratio and decoder_conf tr_conv_group_ratio
     * (seanet_encoder.py:224,234,321; seanet_decoder.py:219,229,324): groups = channels / 2 / ratio; <= 0: dense */
    int32_t conv_group_ratio;
    int32_t tr_conv_group_ratio;
    /* time-domain stacks (arch 0): residual blocks per stage and their dilation base -- block j's first conv has dilation
     * dilation_base^j (seanet_encoder.py:122-128, seanet_decoder.py:141-147; the soundstream_noncausal YAMLs use 3 and 2).
     * 0 in either field selects the reference defaults (1 block, base 2). */
    int32_t n_residual_layers;
    int32_t dilation_base;
    /* encoder_conf / decoder_conf `norm` (conv.py:21-55) for arch 0 -- 0: time_group_norm (GroupNorm(1, C) after every conv),
     * 1: weight_norm (tensors `...weight_g` / `...weight_v`, folded at fcb_finalize; a folded `...weight` is accepted too),
     * 2: none.  `causal` (0 / 1): left-only reflect padding of the convs and right-only trimming of the transposed convs
     * (conv.py:251-253,293-297; trim_right_ratio 1) -- conf/soundstream_16k_n32_600k_step.yaml is {weight_norm, causal}.
     * causal with time_group_norm is refused like the reference does (conv.py:46-47); arch 1 takes neither. */
    int32_t norm;
    int32_t causal;
    /* Audio channels of the time-domain stacks (arch 0): 0 or 1 mono, 2 stereo (Encodec input_size / SEANetDecoder channels;
     * _encode asserts 0 < channels <= 2, codec_basic.py:342-344).  A stereo handle takes and returns every waveform buffer in
     * the reference's channel-planar layout [B, 2, L]; the RMS scale is one value per clip, taken from the mono mix
     * x.mean(dim=1) (:366-369).  The first encoder conv then has 2 input channels ("encoder.model.0.conv.conv.weight"
     * [n_filters, 2, k]) and the last decoder conv 2 output channels (weight [2, n_filters, k], bias and GroupNorm affine [2]).
     * arch 1 (FreqCodec, which STFTs x.squeeze(1)) is mono only: fcb_create refuses channels 2 there. */
    int32_t channels;
} fcb_config;

typedef struct fcb_handle fcb_handle;

/* Library / build identification ("funcodec_b200 x.y sm_100a"). */
FCB_API const char* fcb_version(void);

/* Create a model instance bound to the current CUDA device.  Replaces the module construction in
 * GANSpeechCodecTask.build_model (gan_speech_codec.py:319-343). */
FCB_API int fcb_create(const fcb_config* cfg, fcb_handle** out);

/* Feed one tensor of the reference state_dict (names per SURVEY.md App. D, e.g.
 * "encoder.model.0.conv.conv.weight", "decoder.model.3.convtr.convtr.weight",
 * "encoder.model.16.lstm.weight_ih_l0", "quantizer.rq.model.embed").  `data` is a HOST pointer to
 * contiguous fp32; the library copies it.  Unknown names are ignored with return 1 (mirrors
 * filter_state_dict, funcodec/torch_utils/load_pretrained_model.py:12-43); shape mismatches are errors.
 * Replaces load_state_dict in AbsTask.build_model_from_file (funcodec/tasks/abs_task.py:1939-1944). */
FCB_API int fcb_set_tensor(fcb_handle* h, const char* name, const float* data, int32_t ndim, const int64_t* shape);

/* Repack weights for the kernels, upload, precompute |c|^2.  Synchronous. */
FCB_API int fcb_finalize(fcb_handle* h);

/* T' for a clip of L samples: ceil(L / hop). */
FCB_API int fcb_num_frames(const fcb_handle* h, int32_t L);
/* Samples the decoder produces for n_frames codec frames: T'*hop (arch 0) or stft_hop*(T'*prod(time ratios) - 1)
 * (arch 1, torch.istft with center=True).  fcb_decode_* accept out_len <= this. */
FCB_API int fcb_decoded_length(const fcb_handle* h, int32_t n_frames);
/* n_q for a target bandwidth (<=0: all), ResidualVectorQuantizer.get_num_quantizers_for_bandwidth
 * (funcodec/modules/quantization/vq.py:105-112). */
FCB_API int fcb_num_quantizers_for_bandwidth(const fcb_handle* h, double bandwidth);

/* Encodec.inference_encoding (codec_basic.py:720-764) / the encode half of Encodec.inference:
 * RMS-normalise (:366-371) -> SEANetEncoder -> RVQ (ddp_core_vq.py:367-418).
 *   wav          dev [B, L] fp32 ([B, 2, L] stereo)
 *   codes        dev [n_q, B, T'] int64                               (required)
 *   quant        dev [B, T', D] fp32 quantized embeddings            (nullable)
 *   scale        dev [B] fp32 per-clip RMS scale (1.0 when !audio_normalize)   (nullable)
 *   sub_quants   dev [n_q, B, D, T'] fp32                            (nullable)
 *   encoder_out  dev [B, T', D] fp32 un-quantized encoder output     (nullable; parity/debug) */
FCB_API int fcb_encode(fcb_handle* h, const float* wav, int32_t B, int32_t L, int32_t n_q,
               int64_t* codes, float* quant, float* scale, float* sub_quants, float* encoder_out,
               void* stream);

/* Encodec.inference_decoding_emb (codec_basic.py:804-836) and the decode half of Encodec.inference
 * (:709-711): SEANetDecoder -> optional * scale -> keep the first out_len samples.
 *   emb dev [B, T', D]; scale dev [B] or NULL; wav_out dev [B, out_len] ([B, 2, out_len] stereo), out_len <= T' * hop. */
FCB_API int fcb_decode_emb(fcb_handle* h, const float* emb, int32_t B, int32_t n_frames, const float* scale,
                   float* wav_out, int32_t out_len, void* stream);

/* Encodec.inference_decoding (codec_basic.py:766-802): codes dev [B, T', n_q] int64 ->
 * sum_q embed[q][code] (ddp_core_vq.py:442-453) -> decoder.  emb_out dev [B, T', D] nullable. */
FCB_API int fcb_decode_codes(fcb_handle* h, const int64_t* codes, int32_t B, int32_t n_frames, int32_t n_q,
                     float* emb_out, float* wav_out, int32_t out_len, void* stream);

/* Deferred data errors.  fcb_decode_codes validates token ids ON THE DEVICE (a token < 0 or >= codebook_size is skipped and
 * raises a sticky flag) so that the call stays asynchronous; the reference's F.embedding raises for such a token
 * (ddp_core_vq.py:190-192, e.g. the -1 quantize-dropout indices or a codecs.txt of a larger codebook).  fcb_check_errors
 * synchronises `stream`, reads and clears the flag and returns FCB_E_INVALID (with fcb_last_error text) when any call since the
 * previous check saw an out-of-range token.  B200Encodec.inference_decoding calls it and raises IndexError. */
FCB_API int fcb_check_errors(fcb_handle* h, void* stream);

/* Encodec.inference (codec_basic.py:670-718) with need_recon=True in one call: fcb_encode followed by
 * decode of the quantized embeddings, recon dev [B, L] ([B, 2, L] stereo).  use_scale as in the reference. */
FCB_API int fcb_roundtrip(fcb_handle* h, const float* wav, int32_t B, int32_t L, int32_t n_q, int32_t use_scale,
                  int64_t* codes, float* quant, float* scale, float* sub_quants, float* recon,
                  void* stream);

/* Same as fcb_roundtrip but with HOST buffers (pinned for real asynchrony): the library stages the
 * H2D copy of wav and the D2H copies of codes/recon on `stream` and synchronises it before returning.
 * This is the call a non-PyTorch host (the drop-in CLI worker) makes. */
FCB_API int fcb_roundtrip_host(fcb_handle* h, const float* wav_host, int32_t B, int32_t L, int32_t n_q,
                       int32_t use_scale, int64_t* codes_host, float* recon_host, void* stream);

/* ---- segment_dur != None (Encodec.segment_length / segment_stride / _encode / _decode, codec_basic.py:287-298,334-359,
 * 382-396; _linear_overlap_add :77-116).  The clip is cut at offsets 0, stride, 2*stride, ... < L into segments of
 * seg_len samples (the last ones shorter); every segment is normalised, encoded, quantized and decoded on its own and
 * the decoded segments are cross-faded.  seg_len = int(segment_dur * sample_rate),
 * stride = max(1, int((1 - overlap_ratio) * seg_len)) are computed by the caller exactly like the reference properties.
 * The n_full full-length segments run as ONE batch of n_full*B clips (clip index s*B + b); the n_tail shorter trailing
 * segments run one by one.  Time-domain Encodec (arch 0) only. */
#define FCB_MAX_TAIL_SEGMENTS 16
typedef struct fcb_segment_plan {
    int32_t n_seg, n_full, n_tail;       /* n_seg = n_full + n_tail = len(range(0, L, stride)) */
    int32_t frames_full, decoded_full;   /* T' and T'*hop of a full segment */
    int32_t tail_len[FCB_MAX_TAIL_SEGMENTS], tail_frames[FCB_MAX_TAIL_SEGMENTS];
    int64_t total_frames;                /* n_full*frames_full + sum(tail_frames): frames per clip over all segments */
} fcb_segment_plan;
/* Fails (FCB_E_INVALID) when the reference would: more than FCB_MAX_TAIL_SEGMENTS short segments, or a non-final decoded
 * segment ending after the final one (the reference's overlap-add raises a size mismatch there, codec_basic.py:112). */
FCB_API int fcb_plan_segments(fcb_handle* h, int32_t L, int32_t seg_len, int32_t stride, fcb_segment_plan* plan);
/* The same arithmetic without a handle or a device (hop = samples per codec frame): host-side planning and the CPU tests. */
FCB_API int fcb_plan_segments_for_hop(int32_t hop, int32_t L, int32_t seg_len, int32_t stride, fcb_segment_plan* plan);
/* Encodec.inference with segments.  Outputs (dev), full segments first then the tails in order:
 *   codes  int64: [n_q][n_full*B][frames_full] followed, per tail i, by [n_q][B][tail_frames[i]]
 *   quant  fp32 or NULL: [n_full*B][frames_full][D] followed by [B][tail_frames[i]][D] per tail
 *   scale  fp32 or NULL: [n_seg][B]
 *   recon  fp32 or NULL: [B][L], [B][2][L] stereo (NULL = encode only, Encodec.inference_encoding)
 * wav is [B][L] ([B][2][L] stereo); every segment of a stereo clip gets one scale from its mono mix. */
FCB_API int fcb_roundtrip_segmented(fcb_handle* h, const float* wav, int32_t B, int32_t L, int32_t seg_len, int32_t stride,
                                    int32_t n_q, int32_t use_scale, int64_t* codes, float* quant, float* scale,
                                    float* recon, void* stream);

/* Number of kernels this handle has launched since creation (bench.py's gpu_launches). */
FCB_API int64_t fcb_launch_count(const fcb_handle* h);
/* Enable/disable per-phase device timing (CUDA events on `stream`); phase ids FCB_PHASE_*. */
#define FCB_PHASE_ENCODER_CONV 0
#define FCB_PHASE_ENCODER_LSTM 1
#define FCB_PHASE_RVQ          2
#define FCB_PHASE_DECODER_LSTM 3
#define FCB_PHASE_DECODER_CONV 4
#define FCB_NUM_PHASES         5
FCB_API int fcb_set_profiling(fcb_handle* h, int32_t enabled);
/* Milliseconds spent per phase in the most recent call (synchronises the recorded events). */
FCB_API int fcb_get_phase_ms(fcb_handle* h, float* ms_out /* [FCB_NUM_PHASES] */);

/* Options (integer valued): "use_tc" 1/0 -- tensor-core (tcgen05) conv path vs fp32 SIMT path; must be set
 * before fcb_finalize to enable, may be cleared at any time.  Env FCB_DISABLE_TC=1 sets the default to 0. */
/* "use_tc2d" (FreqCodec, arch 1): bit mask of the 2-D layer classes that run on the tensor-core path -- 1: C_in % 32 == 0,
 * 2: C_in < 32 (several frequency taps per 32-channel chunk), 4: C_out padded to 16 (the 32 -> 3 output conv); default 7,
 * 0 = every 2-D conv on the fp32 SIMT kernel.  May be changed at any time; env FCB_USE_TC2D=<mask> sets the default. */
/* "stft_tc" 1/0 (default 1; env FCB_STFT_TC): STFT / iSTFT of the FreqCodec front / back end as two tensor-core GEMMs (windowed
 * DFT bases as conv weight images; needs n_fft and hop to be multiples of 32) instead of the direct-DFT kernels.
 * "conv2d_small_cout" 1/0 (default 1; env FCB_CONV2D_SMALL_COUT): halo-tile SIMT kernel for 2-D convs with C_out <= 4 (FreqCodec's
 * 32 -> 3 output conv) instead of the padded tensor-core n-tile.  Both were validated and A/B-timed on a B200 in round 2
 * (profiles/ab_bringup_r2a.txt). */
FCB_API int fcb_set_option(fcb_handle* h, const char* key, int32_t value);

/* TEST HOOK (tests/test_gpu_layers.py): run ONE packed conv layer, addressed by its reference module prefix
 * ("encoder.model.3", "decoder.model.3", "encoder.model.1.block.1", "encoder.model.16.lstm.ih0", ...), on a plain
 * channels-last input x dev [B][T][C_in] (optional ELU on load; "encoder.model.0" of a stereo handle reads x channel-planar
 * [B][2][T] like fcb_encode's waveform).  y dev receives the RAW output (bias added,
 * GroupNorm not applied) as [B][t_out][c_out] where for a transposed conv t_out is the UNtrimmed length and
 * row_off the first kept row (conv.py:299-303); stats dev [B][2] = (mean, rstd) of the layer's GroupNorm or NULL. */
FCB_API int fcb_debug_conv1d(fcb_handle* h, const char* layer, const float* x, int32_t B, int32_t T, int32_t elu,
                             float* y, int64_t y_capacity, float* stats, int32_t* t_out, int32_t* c_out,
                             int32_t* row_off, void* stream);

/* TEST HOOK (tests/test_gpu_freq.py), FreqCodec 2-D layers: x dev [B][F][T][C_store] plain channels-last input where
 * C_store is the layer's stored input channel count (returned in dims[7]; 4 for "encoder.model.0": 3 features + one zero
 * channel).  y dev receives the RAW output [B][F_raw][T_raw][C]; dims[8] = {F_raw, T_raw, C, f_off, t_off, F, T, C_store}:
 * the logical window of a transposed conv is rows f_off..f_off+F-1, columns t_off..t_off+T-1 (unpad2d, conv.py:430-445);
 * GroupNorm statistics cover the whole raw tensor. */
FCB_API int fcb_debug_conv2d(fcb_handle* h, const char* layer, const float* x, int32_t B, int32_t F, int32_t T, int32_t elu,
                             float* y, int64_t y_capacity, float* stats, int32_t* dims /* [8] */, void* stream);

FCB_API const char* fcb_last_error(const fcb_handle* h);
FCB_API void fcb_destroy(fcb_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* FUNCODEC_B200_H_ */
