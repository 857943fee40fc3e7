"""Python host side of the drop-in: the reference's `Encodec` inference interface on top of the C ABI.

`B200Encodec` mirrors the METHOD SEAM funcodec/bin/codec_inference.py uses on the model object
(SURVEY.md §8(b)): `inference`, `inference_encoding`, `inference_decoding`, `inference_decoding_emb`
(/root/reference/funcodec/models/codec_basic.py:670-836) with the same argument names, return-dict keys,
tensor layouts and error behaviour, plus the `.quantizer.{sampling_rate, encoder_hop_length, codebook_size}`
attributes Speech2Token reads (codec_inference.py:121,362,365).  PyTorch is only the allocator / stream
provider here: every FLOP runs in funcodec_b200/lib/libfuncodec_b200.so.
"""
import ctypes
from typing import Dict, List, Optional

import torch

from . import _capi
from .config import CodecConfig, NORM_CODES


class _QuantizerInfo:
    """The attributes of CostumeQuantizer that callers read (costume_quantizer.py:49-53)."""

    def __init__(self, cfg: CodecConfig):
        self.sampling_rate = cfg.sample_rate
        self.encoder_hop_length = cfg.hop_length
        self.codebook_size = cfg.codebook_size
        self.code_dim = cfg.dimension
        self.num_quantizers = cfg.num_quantizers

    def output_size(self):
        return self.code_dim


def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


class B200Encodec:
    """Inference-only stand-in for funcodec.models.codec_basic.Encodec backed by the CUDA library."""

    def __init__(self, cfg: CodecConfig, state_dict: Dict[str, torch.Tensor], device: str = "cuda:0",
                 options: Optional[Dict[str, int]] = None, segment_dur: Optional[float] = None,
                 overlap_ratio: Optional[float] = None):
        self.cfg = cfg
        # Encodec(segment_dur=, overlap_ratio=) (codec_basic.py:143-144,218-219); the shipped YAMLs set both to null
        self.segment_dur = segment_dur
        self.overlap_ratio = overlap_ratio
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _capi.FcbError("B200Encodec needs a CUDA device; there is no CPU path")
        self._lib = _capi.load_library()
        self.quantizer = _QuantizerInfo(cfg)
        self.sample_rate = cfg.sample_rate
        self.audio_normalize = cfg.audio_normalize
        c = _capi.FcbConfig()
        c.n_ratios = len(cfg.ratios)
        for i, r in enumerate(cfg.ratios):
            c.ratios[i] = r
        c.n_filters, c.dimension = cfg.n_filters, cfg.dimension
        c.kernel_size, c.last_kernel_size, c.residual_kernel_size = cfg.kernel_size, cfg.last_kernel_size, cfg.residual_kernel_size
        c.lstm_layers, c.codebook_size, c.num_quantizers = cfg.lstm_layers, cfg.codebook_size, cfg.num_quantizers
        c.sample_rate, c.audio_normalize, c.gn_eps = cfg.sample_rate, int(cfg.audio_normalize), cfg.gn_eps
        c.arch, c.n_fft, c.stft_hop = cfg.arch, cfg.n_fft, cfg.stft_hop
        c.conv_group_ratio, c.tr_conv_group_ratio = cfg.conv_group_ratio, cfg.tr_conv_group_ratio
        c.n_residual_layers, c.dilation_base = cfg.n_residual_layers, cfg.dilation_base
        c.norm, c.causal = NORM_CODES[cfg.norm], int(cfg.causal)
        c.channels = cfg.channels
        for i, r in enumerate(cfg.ratios_f):
            c.ratios_f[i] = r
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            rc = self._lib.fcb_create(ctypes.byref(c), ctypes.byref(self._h))
            if rc != 0:
                why = " (stereo is built for the time-domain Encodec only)" if cfg.channels == 2 and cfg.arch != 0 else ""
                raise _capi.FcbError(f"fcb_create failed (rc={rc}){why}")
            for key, val in (options or {}).items():
                _capi.check(self._lib, self._h, self._lib.fcb_set_option(self._h, key.encode(), int(val)),
                            f"fcb_set_option({key})")
            for name, t in state_dict.items():
                if not t.is_floating_point():
                    continue
                t = t.detach().to("cpu", torch.float32).contiguous()
                shape = (ctypes.c_int64 * max(t.dim(), 1))(*t.shape)
                _capi.check(self._lib, self._h, self._lib.fcb_set_tensor(self._h, name.encode(), _ptr(t), t.dim(), shape),
                            f"fcb_set_tensor({name})")
            _capi.check(self._lib, self._h, self._lib.fcb_finalize(self._h), "fcb_finalize")

    # ------------------------------------------------------------------ nn.Module-ish surface used by the CLI
    def eval(self):
        return self

    def to(self, *args, **kwargs):
        return self

    def __del__(self):
        h, lib = getattr(self, "_h", None), getattr(self, "_lib", None)
        if h and lib:
            lib.fcb_destroy(h)
            self._h = None

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _ck(self, rc, what):
        return _capi.check(self._lib, self._h, rc, what)

    def num_frames(self, length: int) -> int:
        return self.cfg.frames(length)

    def launch_count(self) -> int:
        return int(self._lib.fcb_launch_count(self._h))

    def set_profiling(self, enabled: bool):
        self._ck(self._lib.fcb_set_profiling(self._h, int(enabled)), "fcb_set_profiling")

    def phase_ms(self) -> Dict[str, float]:
        arr = (ctypes.c_float * _capi.FCB_NUM_PHASES)()
        self._ck(self._lib.fcb_get_phase_ms(self._h, arr), "fcb_get_phase_ms")
        return {n: float(arr[i]) for i, n in enumerate(_capi.PHASE_NAMES)}

    def debug_conv(self, layer: str, x_btc: torch.Tensor, elu: bool = False, want_stats: bool = True):
        """fcb_debug_conv1d test hook: one packed layer on a plain channels-last input -> (raw y [B,t_out,c_out],
        stats [B,2] | None, row_off).  The stereo first conv takes the waveform's planar layout, so x is transposed for it."""
        B, T, Cx = x_btc.shape
        if layer == "encoder.model.0" and Cx > 1:
            x_btc = x_btc.transpose(1, 2)
        x = x_btc.to(self.device, torch.float32).contiguous()
        cap = B * (T + 2) * 8192
        y = torch.empty(cap, dtype=torch.float32, device=self.device)
        stats = torch.empty((B, 2), dtype=torch.float32, device=self.device) if want_stats else None
        t_out, c_out, row_off = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
        with torch.cuda.device(self.device):
            self._ck(self._lib.fcb_debug_conv1d(self._h, layer.encode(), _ptr(x), B, T, int(elu), _ptr(y), cap, _ptr(stats),
                                                ctypes.byref(t_out), ctypes.byref(c_out), ctypes.byref(row_off),
                                                self._stream()), f"fcb_debug_conv1d({layer})")
        n = B * t_out.value * c_out.value
        return y[:n].view(B, t_out.value, c_out.value), stats, row_off.value

    @property
    def segment_length(self) -> Optional[int]:        # codec_basic.py:287-291
        return None if self.segment_dur is None else int(self.segment_dur * self.sample_rate)

    @property
    def segment_stride(self) -> Optional[int]:        # codec_basic.py:293-298
        seg = self.segment_length
        return None if seg is None else max(1, int((1 - self.overlap_ratio) * seg))

    def plan_segments(self, L: int) -> "_capi.FcbSegmentPlan":
        plan = _capi.FcbSegmentPlan()
        self._ck(self._lib.fcb_plan_segments(self._h, L, self.segment_length, self.segment_stride, ctypes.byref(plan)),
                 "fcb_plan_segments")
        return plan

    def _inference_segmented(self, x: torch.Tensor, need_recon: bool, n_q: int, use_scale: bool):
        """Encodec.inference with segment_dur != None (codec_basic.py:334-359,382-396,695-718): one list entry per segment,
        recon_speech = linear overlap-add of the decoded segments trimmed to L.  sub_quants are not produced here."""
        B, L = x.shape[0], x.shape[-1]
        plan = self.plan_segments(L)
        D, dev = self.cfg.dimension, self.device
        nf, T0 = plan.n_full, plan.frames_full
        codes = torch.empty(n_q * B * plan.total_frames, dtype=torch.int64, device=dev)
        quant = torch.empty(B * plan.total_frames * D, dtype=torch.float32, device=dev)
        scale = torch.empty((plan.n_seg, B, 1), dtype=torch.float32, device=dev)
        recon = torch.empty((B, self.cfg.channels, L), dtype=torch.float32, device=dev) if need_recon else None
        with torch.cuda.device(dev):
            self._ck(self._lib.fcb_roundtrip_segmented(self._h, _ptr(x), B, L, self.segment_length, self.segment_stride, n_q,
                                                       int(use_scale), _ptr(codes), _ptr(quant), _ptr(scale), _ptr(recon),
                                                       self._stream()), "fcb_roundtrip_segmented")
        idx, embs = [], []
        with_scale = use_scale and self.audio_normalize
        cfull = codes[:n_q * nf * B * T0].view(n_q, nf, B, T0)
        qfull = quant[:nf * B * T0 * D].view(nf, B, T0, D)
        for s in range(nf):
            idx.append(cfull[:, s])
            embs.append((qfull[s], scale[s] if with_scale else None))
        co, qo = n_q * nf * B * T0, nf * B * T0 * D
        for i in range(plan.n_tail):
            Ti = plan.tail_frames[i]
            idx.append(codes[co:co + n_q * B * Ti].view(n_q, B, Ti))
            embs.append((quant[qo:qo + B * Ti * D].view(B, Ti, D), scale[nf + i] if with_scale else None))
            co += n_q * B * Ti
            qo += B * Ti * D
        return dict(recon_speech=recon, code_indices=idx, code_embeddings=embs, sub_quants=[None] * plan.n_seg)

    def set_option(self, key: str, value: int) -> None:
        """fcb_set_option ("use_tc" may only be cleared after construction; "use_tc2d" may change at any time)."""
        self._ck(self._lib.fcb_set_option(self._h, key.encode(), int(value)), f"fcb_set_option({key})")

    def debug_conv2d(self, layer: str, x_bftc: torch.Tensor, elu: bool = False):
        """fcb_debug_conv2d test hook (FreqCodec): one packed 2-D layer on a plain channels-last input [B,F,T,C] ->
        (raw y [B,F_raw,T_raw,C_out], stats [B,2], (f_off, t_off, F, T) logical window).  Inputs with fewer channels than
        the layer stores (the 3 mag_phase features of encoder.model.0, stored as 4) are zero-padded."""
        x = x_bftc.to(self.device, torch.float32)
        B, F, T, C = x.shape
        dims = (ctypes.c_int32 * 8)()
        c_store = 4 if (layer == "encoder.model.0" and C == 3) else C
        if c_store != C:
            x = torch.cat([x, torch.zeros(B, F, T, c_store - C, device=self.device)], dim=-1)
        x = x.contiguous()
        cap = min(B * (F + 1) * (T + 1) * 4096, 1 << 28)      # >= B * F_raw * T_raw * C_out for every supported layer
        y = torch.empty(cap, dtype=torch.float32, device=self.device)
        stats = torch.empty((B, 2), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            self._ck(self._lib.fcb_debug_conv2d(self._h, layer.encode(), _ptr(x), B, F, T, int(elu), _ptr(y), cap, _ptr(stats),
                                                dims, self._stream()), f"fcb_debug_conv2d({layer})")
        F_raw, T_raw, Co, f_off, t_off, Fl, Tl, cs = [int(v) for v in dims]
        if cs != c_store:
            raise ValueError(f"{layer} stores {cs} input channels, got {c_store}")
        return y[:B * F_raw * T_raw * Co].view(B, F_raw, T_raw, Co), stats, (f_off, t_off, Fl, Tl)

    def _prep_speech(self, speech: torch.Tensor) -> torch.Tensor:
        """-> [B, L] for a mono model, channel-planar [B, 2, L] for a stereo one (the reference's [B, C, L] layout)."""
        if self.cfg.channels == 2:
            if speech.dim() != 3 or speech.shape[1] != 2:
                raise ValueError(f"this model is stereo (input_size: 2): speech must be [B, 2, L], got {tuple(speech.shape)}")
            return speech.to(self.device, torch.float32).contiguous()
        if speech.dim() == 3:
            if speech.shape[1] != 1:
                raise ValueError("only mono input is supported (input_size: 1)")
            speech = speech[:, 0, :]
        if speech.dim() != 2:
            raise ValueError("speech must be [B, L] or [B, 1, L]")
        return speech.to(self.device, torch.float32).contiguous()

    # ------------------------------------------------------------------ the four reference entry points
    @torch.no_grad()
    def inference(self, speech: torch.Tensor, need_recon: bool = True, bit_width: int = None,
                  use_scale: bool = True, need_sub_quants: bool = True, need_encoder_out: bool = False):
        """Encodec.inference (codec_basic.py:670-718).  `need_sub_quants=False` skips the [n_q,B,D,T'] tensor
        (the reference always builds it; codec_inference.py only reads it under --need_sub_quants)."""
        x = self._prep_speech(speech)
        B, L = x.shape[0], x.shape[-1]
        C = self.cfg.channels
        Tf = self.num_frames(L)
        # the reference slices self.layers[:n_q] (ddp_core_vq.py:386): a bandwidth above the maximum uses every stage
        n_q = min(self.cfg.num_quantizers_for_bandwidth(bit_width), self.cfg.num_quantizers)
        if self.segment_dur is not None:
            return self._inference_segmented(x, need_recon, n_q, use_scale)
        D = self.cfg.dimension
        dev = self.device
        codes = torch.empty((n_q, B, Tf), dtype=torch.int64, device=dev)
        quant = torch.empty((B, Tf, D), dtype=torch.float32, device=dev)
        scale = torch.empty((B, 1), dtype=torch.float32, device=dev)
        sub = torch.empty((n_q, B, D, Tf), dtype=torch.float32, device=dev) if need_sub_quants else None
        enc = torch.empty((B, Tf, D), dtype=torch.float32, device=dev) if need_encoder_out else None
        recon = None
        # FreqCodec: the iSTFT yields stft_hop * (T_s - 1) samples, possibly fewer than L (the reference's [:, :, :L] slice
        # then simply returns what exists, codec_freq.py:709)
        Lr = min(L, self.cfg.decoded_length(Tf))
        with torch.cuda.device(dev):
            if need_recon and not need_encoder_out and Lr == L:
                recon = torch.empty((B, C, L), dtype=torch.float32, device=dev)
                self._ck(self._lib.fcb_roundtrip(self._h, _ptr(x), B, L, n_q, int(use_scale), _ptr(codes), _ptr(quant),
                                                 _ptr(scale), _ptr(sub), _ptr(recon), self._stream()), "fcb_roundtrip")
            else:
                self._ck(self._lib.fcb_encode(self._h, _ptr(x), B, L, n_q, _ptr(codes), _ptr(quant), _ptr(scale),
                                              _ptr(sub), _ptr(enc), self._stream()), "fcb_encode")
                if need_recon:
                    recon = torch.empty((B, C, Lr), dtype=torch.float32, device=dev)
                    sc = scale if (use_scale and self.audio_normalize) else None
                    self._ck(self._lib.fcb_decode_emb(self._h, _ptr(quant), B, Tf, _ptr(sc), _ptr(recon), Lr,
                                                      self._stream()), "fcb_decode_emb")
        ret_scale = scale if (use_scale and self.audio_normalize) else None
        out = dict(recon_speech=recon, code_indices=[codes], code_embeddings=[(quant, ret_scale)],
                   sub_quants=[sub])
        if need_encoder_out:
            out["encoder_out"] = enc
        return out

    @torch.no_grad()
    def inference_encoding(self, speech: torch.Tensor, need_recon: bool = False, bit_width: int = None,
                           use_scale: bool = True, need_sub_quants: bool = True):
        """Encodec.inference_encoding (codec_basic.py:720-764)."""
        return self.inference(speech, need_recon=need_recon, bit_width=bit_width, use_scale=use_scale,
                              need_sub_quants=need_sub_quants)

    @torch.no_grad()
    def inference_decoding(self, token_idx: torch.Tensor, need_recon: bool = True, bit_width: int = None,
                           use_scale: bool = True):
        """Encodec.inference_decoding (codec_basic.py:766-802): token_idx [B, T', n_q] int64."""
        if token_idx.dim() != 3:
            raise ValueError("token_idx must be [B, T', n_q]")
        tok = token_idx.to(self.device, torch.int64).contiguous()
        B, Tf, n_q = tok.shape
        D, Lo = self.cfg.dimension, self.cfg.decoded_length(Tf)
        emb = torch.empty((B, Tf, D), dtype=torch.float32, device=self.device)
        recon = torch.empty((B, self.cfg.channels, Lo), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            self._ck(self._lib.fcb_decode_codes(self._h, _ptr(tok), B, Tf, n_q, _ptr(emb), _ptr(recon), Lo,
                                                self._stream()), "fcb_decode_codes")
            # out-of-range tokens: F.embedding raises in the reference (ddp_core_vq.py:190-192); here the device flags them
            if self._lib.fcb_check_errors(self._h, self._stream()) < 0:
                raise IndexError(self._lib.fcb_last_error(self._h).decode())
        return dict(recon_speech=recon if need_recon else None, code_indices=None,
                    code_embeddings=[(emb, None)], sub_quants=None)

    @torch.no_grad()
    def inference_decoding_emb(self, token_idx: torch.Tensor, need_recon: bool = True, bit_width: int = None,
                               use_scale: bool = True):
        """Encodec.inference_decoding_emb (codec_basic.py:804-836): token_idx is [B, T', D] embeddings."""
        if token_idx.dim() != 3 or token_idx.shape[-1] != self.cfg.dimension:
            raise ValueError("token_idx must be [B, T', D] embeddings")
        emb = token_idx.to(self.device, torch.float32).contiguous()
        B, Tf, _ = emb.shape
        Lo = self.cfg.decoded_length(Tf)
        recon = None
        if need_recon:
            recon = torch.empty((B, self.cfg.channels, Lo), dtype=torch.float32, device=self.device)
            with torch.cuda.device(self.device):
                self._ck(self._lib.fcb_decode_emb(self._h, _ptr(emb), B, Tf, None, _ptr(recon), Lo,
                                                  self._stream()), "fcb_decode_emb")
        return dict(recon_speech=recon, code_indices=None, code_embeddings=[(emb, None)], sub_quants=None)

    # ------------------------------------------------------------------ host-buffer end-to-end call (bench e2e)
    @torch.no_grad()
    def roundtrip_host(self, wav_pinned: torch.Tensor, codes_pinned: torch.Tensor, recon_pinned: torch.Tensor,
                       bit_width: int = None, use_scale: bool = True):
        """fcb_roundtrip_host: HOST (pinned) buffers in and out, copies inside the call, synchronous.  wav / recon are
        [B, L] (mono) or [B, 2, L] (stereo)."""
        B, L = wav_pinned.shape[0], wav_pinned.shape[-1]
        assert wav_pinned.numel() == B * self.cfg.channels * L and recon_pinned.numel() == wav_pinned.numel()
        n_q = min(self.cfg.num_quantizers_for_bandwidth(bit_width), self.cfg.num_quantizers)
        assert codes_pinned.shape == (n_q, B, self.num_frames(L)) and codes_pinned.dtype == torch.int64
        assert recon_pinned.shape[0] == B and recon_pinned.shape[-1] == L
        with torch.cuda.device(self.device):
            self._ck(self._lib.fcb_roundtrip_host(self._h, _ptr(wav_pinned), B, L, n_q, int(use_scale),
                                                  _ptr(codes_pinned), _ptr(recon_pinned), self._stream()),
                     "fcb_roundtrip_host")
