"""Model hyper-parameters for the codec hot path (host logic, no CUDA).

Mirrors the YAML keys the reference feeds to GANSpeechCodecTask.build_model
(/root/reference/funcodec/tasks/gan_speech_codec.py:301-358): `encoder_conf`, `quantizer_conf`,
`decoder_conf`, `model_conf` of egs/LibriTTS/codec/conf/encodec_16k_n32_600k_step{,_ds640}.yaml.
Representable: norm time_group_norm / weight_norm / none, causal or not (time-domain stacks), true_skip=False, compress=2,
LSTM or no sequence model, stacked dilated residual blocks, RVQ without projections, mono or stereo time-domain audio.
"""
from dataclasses import dataclass, field, asdict
from typing import Dict, Optional, Tuple
import math


@dataclass(frozen=True)
class CodecConfig:
    name: str = "encodec_16k_n32_ds640"
    ratios: Tuple[int, ...] = (8, 5, 4, 2, 2)   # encoder_conf.ratios / decoder_conf.ratios
    n_filters: int = 32                          # SEANetEncoder default (seanet_encoder.py:90)
    dimension: int = 128                         # model_conf.odim / quantizer input_size
    kernel_size: int = 7
    last_kernel_size: int = 7
    residual_kernel_size: int = 3
    lstm_layers: int = 2                         # seq_layer_num default
    codebook_size: int = 1024                    # quantizer_conf.codebook_size
    num_quantizers: int = 32                     # quantizer_conf.num_quantizers
    sample_rate: int = 16000                     # quantizer_conf.sampling_rate / target_sample_hz
    audio_normalize: bool = True                 # model_conf.audio_normalize
    gn_eps: float = 1e-5                         # nn.GroupNorm default
    # FreqCodec variant (funcodec/models/codec_freq.py, codec_domain ['mag_phase', 'mag_phase']): arch = 1, `ratios` are then
    # the TIME ratios and `ratios_f` the FREQUENCY ratios of encoder_conf.ratios [[f, t], ...]
    arch: int = 0
    ratios_f: Tuple[int, ...] = ()
    n_fft: int = 512
    stft_hop: int = 160
    # grouped 2-D convs (encoder_conf / decoder_conf `conv_group_ratio`, decoder_conf `tr_conv_group_ratio`;
    # seanet_encoder.py:224,234,321, seanet_decoder.py:219,229,324): groups = channels // 2 // ratio, -1 = dense
    conv_group_ratio: int = -1
    tr_conv_group_ratio: int = -1
    # residual blocks per stage / dilation base of the time-domain stacks (encoder_conf / decoder_conf n_residual_layers,
    # dilation_base; seanet_encoder.py:122-128): block j's first conv has dilation dilation_base ** j
    n_residual_layers: int = 1
    dilation_base: int = 2
    # encoder_conf / decoder_conf `norm` and `causal` of the time-domain stacks (conv.py:21-55,251-253,293-297):
    # 'time_group_norm' | 'weight_norm' | 'none'; causal needs a norm other than time_group_norm (conv.py:46-47)
    norm: str = "time_group_norm"
    causal: bool = False
    # audio channels of the time-domain stacks: top-level `input_size` / decoder_conf `channels` (seanet_encoder.py:91-110,
    # seanet_decoder.py:89-161); 2 = stereo, waveforms [B, 2, L] (codec_basic.py:342-344 allows 1 or 2).  FreqCodec is mono.
    channels: int = 1

    def conv_groups(self, channels: int) -> int:
        """groups of a 2-D conv whose reference expression is `channels // 2 // conv_group_ratio`."""
        return channels // 2 // self.conv_group_ratio if self.conv_group_ratio > 0 else 1

    def tr_conv_groups(self, channels: int) -> int:
        return channels // 2 // self.tr_conv_group_ratio if self.tr_conv_group_ratio > 0 else 1

    @property
    def hop_length(self) -> int:
        h = int(math.prod(self.ratios))
        return h * self.stft_hop if self.arch == 1 else h

    @property
    def top_channels(self) -> int:
        return self.n_filters * (2 ** len(self.ratios))

    def frames(self, length: int) -> int:
        if self.arch == 1:                       # STFT frames (center=True) then the encoder's time strides
            ts, tp = 1 + length // self.stft_hop, int(math.prod(self.ratios))
            return -(-ts // tp)
        return -(-length // self.hop_length)

    def decoded_length(self, n_frames: int) -> int:
        if self.arch == 1:                       # torch.istft(center=True, length=None)
            return self.stft_hop * (n_frames * int(math.prod(self.ratios)) - 1)
        return n_frames * self.hop_length

    def bandwidth_per_quantizer(self) -> float:
        """ResidualVectorQuantizer.get_bandwidth_per_quantizer (funcodec/modules/quantization/vq.py:114-117)."""
        return math.log2(self.codebook_size) * self.sample_rate / self.hop_length

    def num_quantizers_for_bandwidth(self, bandwidth: Optional[float]) -> int:
        """vq.py:105-112."""
        n_q = self.num_quantizers
        if bandwidth and bandwidth > 0.0:
            n_q = int(max(1, math.floor(bandwidth / self.bandwidth_per_quantizer())))
        return n_q

    def to_dict(self) -> Dict:
        return asdict(self)


PRESETS: Dict[str, CodecConfig] = {
    # BASELINE.json configs 1, 2, 5
    "encodec_16k_n32_ds640": CodecConfig(),
    # BASELINE.json config 3
    "encodec_16k_n32_ds320": CodecConfig(name="encodec_16k_n32_ds320", ratios=(8, 5, 4, 2)),
    # small shapes for parity tests (same topology, every kernel family exercised)
    "tiny_ds40": CodecConfig(name="tiny_ds40", ratios=(5, 4, 2), n_filters=8, dimension=32,
                             codebook_size=64, num_quantizers=8),
    # BASELINE.json config 4: repo YAML conf/freqcodec_mag_phase_16k_n32_600k_step.yaml (ratios [[4,1],[4,1],[4,2],[4,1]],
    # conv groups = 1 -- the hub model's gr8 grouping is not in the repository, SURVEY.md §6)
    "freqcodec_magphase_16k_n32_ds320": CodecConfig(name="freqcodec_magphase_16k_n32_ds320", arch=1, ratios=(1, 1, 2, 1),
                                                    ratios_f=(4, 4, 4, 4)),
    # repo YAML conf/freqcodec_mag_phase_16k_n32_600k_step_ds640.yaml (ratios [[4, 2], [4, 1], [4, 2], [4, 1]], hop 640)
    "freqcodec_magphase_16k_n32_ds640": CodecConfig(name="freqcodec_magphase_16k_n32_ds640", arch=1, ratios=(2, 1, 2, 1),
                                                    ratios_f=(4, 4, 4, 4)),
    "freq_small_ds640": CodecConfig(name="freq_small_ds640", arch=1, ratios=(2, 1, 2, 1), ratios_f=(4, 4, 4, 4), n_filters=4,
                                    dimension=32, codebook_size=64, num_quantizers=6),
    # the hub checkpoint BASELINE config 4 names ("...gr8nq32ds320"): conv_group_ratio 8 in the resblocks / downsampling convs;
    # its YAML is not in the repository (SURVEY.md §6), so the transposed convs are assumed grouped alike
    "freqcodec_magphase_16k_n32_ds320_gr8": CodecConfig(name="freqcodec_magphase_16k_n32_ds320_gr8", arch=1, ratios=(1, 1, 2, 1),
                                                        ratios_f=(4, 4, 4, 4), conv_group_ratio=8, tr_conv_group_ratio=8),
    "freq_small_grouped": CodecConfig(name="freq_small_grouped", arch=1, ratios=(1, 1, 2, 1), ratios_f=(4, 4, 4, 4), n_filters=8,
                                      dimension=32, codebook_size=64, num_quantizers=6, conv_group_ratio=1, tr_conv_group_ratio=2),
    "freq_small": CodecConfig(name="freq_small", arch=1, ratios=(1, 1, 2, 1), ratios_f=(4, 4, 4, 4), n_filters=4,
                              dimension=32, codebook_size=64, num_quantizers=6),
    # conf/soundstream_noncausal_16k_n32_600k_step{,_ds640}.yaml: 3 dilated residual blocks per stage, no sequence model, D = 512
    "soundstream_noncausal_16k_n32_ds320": CodecConfig(name="soundstream_noncausal_16k_n32_ds320", ratios=(8, 5, 4, 2), dimension=512,
                                                       lstm_layers=0, n_residual_layers=3),
    "soundstream_noncausal_16k_n32_ds640": CodecConfig(name="soundstream_noncausal_16k_n32_ds640", ratios=(8, 5, 4, 2, 2), dimension=512,
                                                       lstm_layers=0, n_residual_layers=3),
    "soundstream_noncausal_small": CodecConfig(name="soundstream_noncausal_small", ratios=(5, 4, 2), n_filters=4, dimension=48,
                                               codebook_size=64, num_quantizers=4, lstm_layers=0, n_residual_layers=3,
                                               audio_normalize=False),
    # conf/soundstream_16k_n32_600k_step.yaml: weight_norm, causal, 3 dilated residual blocks per stage, no sequence model
    "soundstream_16k_n32_ds320": CodecConfig(name="soundstream_16k_n32_ds320", ratios=(8, 5, 4, 2), dimension=512, lstm_layers=0,
                                             n_residual_layers=3, norm="weight_norm", causal=True),
    "soundstream_causal_small": CodecConfig(name="soundstream_causal_small", ratios=(5, 4, 2), n_filters=4, dimension=48,
                                            codebook_size=64, num_quantizers=4, lstm_layers=0, n_residual_layers=3,
                                            norm="weight_norm", causal=True),
    # weight_norm with the SLSTM kept, non-causal (every norm / sequence-model combination shares the same kernels)
    "weightnorm_lstm_small": CodecConfig(name="weightnorm_lstm_small", ratios=(5, 4, 2), n_filters=8, dimension=32,
                                         codebook_size=64, num_quantizers=8, norm="weight_norm"),
    "small_ds320": CodecConfig(name="small_ds320", ratios=(8, 5, 4, 2), n_filters=8, dimension=64,
                               codebook_size=256, num_quantizers=8),
    # the 48 kHz stereo layout seanet_encoder.py:63-65 names ("48HZ -> channels = 2, norm = time_group_norm, causal = False"):
    # hop 320, 150 frames per second
    "encodec_48k_stereo": CodecConfig(name="encodec_48k_stereo", ratios=(8, 5, 4, 2), sample_rate=48000, num_quantizers=16,
                                      channels=2),
    # small stereo shapes for the parity tests: time_group_norm + SLSTM, and weight_norm + causal (no GroupNorm on the last layer)
    "stereo_small": CodecConfig(name="stereo_small", ratios=(5, 4, 2), n_filters=8, dimension=32, codebook_size=64,
                                num_quantizers=8, channels=2),
    "stereo_causal_small": CodecConfig(name="stereo_causal_small", ratios=(5, 4, 2), n_filters=4, dimension=48, codebook_size=64,
                                       num_quantizers=4, lstm_layers=0, n_residual_layers=3, norm="weight_norm", causal=True,
                                       channels=2),
}


NORM_CODES = {"time_group_norm": 0, "weight_norm": 1, "none": 2}     # fcb_config.norm


def get_config(name: str) -> CodecConfig:
    return PRESETS[name]
