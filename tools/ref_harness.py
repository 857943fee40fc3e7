"""Import shims that let the UNMODIFIED reference (/root/reference) run in this container.

Only used by tools/gen_golden.py (fixture generation, in the build container).  Nothing under
tests/, bench.py or the product imports this at run time on the GPU box (/root/reference does not
exist there).

Shims (SURVEY.md §8(c)):
  * `librosa` is missing and only used by the training-loss Audio2Mel (codec_basic.py:18) -> stub module.
  * typeguard 4.x rejects `frontend: torch.nn.Module = None` (codec_basic.py:172) -> no-op check.
  * `multi_spectral_window_powers_of_two=[]` avoids Audio2Mel's hard `.cuda()` (codec_basic.py:45).
"""
import sys
import types

REF_ROOT = "/root/reference"


def import_reference():
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    if "librosa" not in sys.modules:
        lib = types.ModuleType("librosa")
        filt = types.ModuleType("librosa.filters")
        filt.mel = lambda *a, **k: None
        lib.filters = filt
        sys.modules["librosa"] = lib
        sys.modules["librosa.filters"] = filt
    from funcodec.models import codec_basic
    codec_basic.check_argument_types = lambda: True
    from funcodec.models.encoder.seanet_encoder import SEANetEncoder
    from funcodec.models.decoder.seanet_decoder import SEANetDecoder
    from funcodec.models.quantizer.costume_quantizer import CostumeQuantizer
    return codec_basic.Encodec, SEANetEncoder, SEANetDecoder, CostumeQuantizer


def build_reference_encodec(cfg):
    """Mirror of GANSpeechCodecTask.build_model (gan_speech_codec.py:301-358) without the
    discriminator; cfg is a funcodec_b200.config.CodecConfig."""
    import torch
    Encodec, SEANetEncoder, SEANetDecoder, CostumeQuantizer = import_reference()
    channels = getattr(cfg, "channels", 1)       # input_size / decoder_conf.channels (2: stereo)
    enc = SEANetEncoder(input_size=channels, dimension=cfg.dimension, n_filters=cfg.n_filters,
                        ratios=list(cfg.ratios), norm=getattr(cfg, "norm", "time_group_norm"), causal=bool(getattr(cfg, "causal", False)),
                        kernel_size=cfg.kernel_size, last_kernel_size=cfg.last_kernel_size,
                        residual_kernel_size=cfg.residual_kernel_size,
                        seq_layer_num=cfg.lstm_layers, seq_model="lstm" if cfg.lstm_layers > 0 else "none",
                        n_residual_layers=cfg.n_residual_layers, dilation_base=cfg.dilation_base)
    quant = CostumeQuantizer(input_size=cfg.dimension, codebook_size=cfg.codebook_size,
                             num_quantizers=cfg.num_quantizers, ema_decay=0.99, kmeans_init=True,
                             sampling_rate=cfg.sample_rate, quantize_dropout=True,
                             rand_num_quant=[2, 4, 8, 16, 32], use_ddp=True,
                             encoder_hop_length=cfg.hop_length)
    dec = SEANetDecoder(input_size=cfg.dimension, channels=channels, n_filters=cfg.n_filters,
                        ratios=list(cfg.ratios), norm=getattr(cfg, "norm", "time_group_norm"), causal=bool(getattr(cfg, "causal", False)),
                        kernel_size=cfg.kernel_size, last_kernel_size=cfg.last_kernel_size,
                        residual_kernel_size=cfg.residual_kernel_size,
                        seq_layer_num=cfg.lstm_layers, seq_model="lstm" if cfg.lstm_layers > 0 else "none",
                        n_residual_layers=cfg.n_residual_layers, dilation_base=cfg.dilation_base)
    model = Encodec(input_size=channels, odim=cfg.dimension, encoder=enc, quantizer=quant, decoder=dec,
                    discriminator=None, target_sample_hz=cfg.sample_rate,
                    multi_spectral_window_powers_of_two=[], audio_normalize=cfg.audio_normalize,
                    segment_dur=None, overlap_ratio=None)
    return model.eval()
