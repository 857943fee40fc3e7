"""Description of the UNMODIFIED reference's model objects and training YAMLs for the CPU tests of
funcodec_b200.integration / bin.codec_inference (tests/test_capi_symbols.py, tests/test_cli.py), so that those tests
run without the reference installed.  Build container only:  python tools/gen_golden_reference_modules.py

tests/golden/reference_modules.json.gz (gzipped JSON) holds
  models[preset]   the `Encodec` that tools/ref_harness.py builds for the preset: the model / quantizer attributes
                   integration.config_from_reference_model reads, every encoder / decoder submodule as
                   [dotted path, class name, public attributes], and the state_dict as {key: shape};
  rvq_use_ddp_false  {key: shape} of the `use_ddp: false` ResidualVectorQuantization (3 x 32 x 16);
  yaml_conf[file]  egs/LibriTTS/codec/conf/<file> as parsed by yaml.safe_load.
"""
import gzip
import json
import os
import sys

import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
from ref_harness import REF_ROOT, build_reference_encodec, import_reference  # noqa: E402
from funcodec_b200 import get_config  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden", "reference_modules.json.gz")
PRESETS = ("encodec_16k_n32_ds320", "tiny_ds40", "soundstream_noncausal_small", "soundstream_causal_small",
           "weightnorm_lstm_small")


def _plain(v):
    if v is None or isinstance(v, (bool, int, float, str)):
        return True
    return isinstance(v, (list, tuple)) and all(_plain(x) for x in v)


def _attrs(obj):
    return {k: v for k, v in sorted(vars(obj).items()) if not k.startswith("_") and k != "training" and _plain(v)}


def describe_model(m):
    d = dict(attrs={k: getattr(m, k) for k in ("audio_normalize", "segment_dur", "overlap_ratio", "codec_domain", "domain_conf")
                    if hasattr(m, k)},
             quantizer=_attrs(m.quantizer), rq_model=_attrs(m.quantizer.rq.model))
    for side in ("encoder", "decoder"):
        d[side] = [[name, type(mod).__name__, _attrs(mod)] for name, mod in getattr(m, side).named_modules()]
    d["state_dict"] = {k: list(v.shape) for k, v in m.state_dict().items()}
    return d


def main():
    out = dict(models={name: describe_model(build_reference_encodec(get_config(name))) for name in PRESETS})
    import_reference()
    from funcodec.modules.quantization.core_vq import ResidualVectorQuantization
    rvq = ResidualVectorQuantization(num_quantizers=3, dim=16, codebook_size=32, decay=0.99, kmeans_init=True, kmeans_iters=10,
                                     threshold_ema_dead_code=2, quantize_dropout=True, rand_num_quant=[1, 2, 3])
    out["rvq_use_ddp_false"] = {k: list(v.shape) for k, v in rvq.state_dict().items()}
    conf = os.path.join(REF_ROOT, "egs", "LibriTTS", "codec", "conf")
    out["yaml_conf"] = {}
    for fn in sorted(os.listdir(conf)):
        with open(os.path.join(conf, fn)) as f:
            out["yaml_conf"][fn] = yaml.safe_load(f)
    with gzip.GzipFile(OUT, "wb", mtime=0) as f:
        f.write((json.dumps(out, separators=(",", ":"), sort_keys=True) + "\n").encode())
    print(OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
