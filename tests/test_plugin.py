"""The registry drop-in: with the reference on sys.path (the unmodified copy oracle/build_ref.py stages under oracle/_ref)
`neurst_b200.plugin.register()` makes the reference's OWN `build_model` return the
libb200st-backed class, through the `class_or_method_args` branch of registry.build_x (neurst/utils/registry.py:90-102)."""
import os

import pytest
import torch

from oracle import build_ref

# the reference checkout, or the unmodified copy of it that build() stages under oracle/_ref
REF = os.environ.get("NEURST_REFERENCE") or build_ref.reference_root()
needs_ref = pytest.mark.skipif(not REF, reason="no reference tree and no copy staged by oracle/build_ref.py")


def _register():
    from oracle import ref_shim
    ref_shim.install()
    from neurst_b200 import plugin
    return plugin, plugin.register()


@needs_ref
def test_registry_lists_the_b200_classes_and_flags_match_the_reference():
    plugin, names = _register()
    from neurst.utils import registry as REG
    for n in ("B200SpeechTransformer", "b200speechtransformer", "b200_speech_transformer", "B200ST"):
        assert n in REG.REGISTRIES["pt"]["model"], n
    assert "B200TransformerEncoder" in REG.REGISTRIES["pt"]["encoder"]
    assert "B200TransformerDecoder" in REG.REGISTRIES["pt"]["decoder"]
    assert "B200MultiHeadAttention" in REG.REGISTRIES["pt"]["base_layer"]
    # the stock class is still there (new names, no override)
    ref_cls = REG.REGISTRIES["pt"]["model"]["SpeechTransformer"]
    b200_cls = REG.REGISTRIES["pt"]["model"]["B200SpeechTransformer"]
    assert ref_cls is not b200_cls and ref_cls.__module__.startswith("neurst_pt")
    ref_flags = {(f.name, f.dtype, f.default) for f in ref_cls.class_or_method_args()}
    our_flags = {(f.name, f.dtype, f.default) for f in b200_cls.class_or_method_args()}
    assert ref_flags == our_flags, ref_flags ^ our_flags


@needs_ref
def test_build_model_through_the_reference_registry_cpu_side():
    """build_x fills the flag defaults and calls B200SpeechTransformer.new(params, src_meta, trg_meta); without a GPU the
    constructor must fail loudly (no CPU fallback) — and with exactly that error, i.e. the registry plumbing worked."""
    _register()
    from neurst_pt.models import build_model
    from neurst_b200.models import speech_transformer_hparams
    from neurst_b200 import lib as L
    params = dict(speech_transformer_hparams("speech_transformer_s")["model.params"])
    params.pop("encoder.ffn_activation")          # left to the flag default, as a user's yaml would
    args = {"model.class": "B200SpeechTransformer", "model.params": params}
    src_meta = {"audio_feature_dim": 80, "audio_feature_channels": 1}
    trg_meta = {"vocab_size": 8192, "eos_id": 8191, "bos_id": 8190, "unk_id": 8189}
    if torch.cuda.is_available():
        model = build_model(args, src_meta, trg_meta)
        assert type(model).__name__ == "B200SpeechTransformer" and model.args["encoder.ffn_activation"] == "relu"
    else:
        with pytest.raises(L.B200STError, match="CUDA"):
            build_model(args, src_meta, trg_meta)
    with pytest.raises(NotImplementedError):      # unsupported variants raise, like the reference's own ValueErrors
        bad = dict(params); bad["encoder.ffn_activation"] = "gelu"
        build_model({"model.class": "B200SpeechTransformer", "model.params": bad}, src_meta, trg_meta)


@needs_ref
def test_override_points_stock_names_at_the_b200_classes():
    plugin, _ = _register()
    from neurst.utils import registry as REG
    saved = {k: dict(v) for k, v in REG.REGISTRIES["pt"].items()}
    try:
        plugin.register(override=True)
        assert REG.REGISTRIES["pt"]["model"]["SpeechTransformer"].__name__ == "B200SpeechTransformer"
        assert REG.REGISTRIES["pt"]["encoder"]["TransformerEncoder"].__name__ == "B200TransformerEncoder"
    finally:
        for k, v in saved.items():
            REG.REGISTRIES["pt"][k].clear(); REG.REGISTRIES["pt"][k].update(v)


@pytest.mark.gpu
def test_plugin_class_forward_on_gpu_without_the_reference():
    """The class factory of the plug-in around a stand-in registry base class (same constructor contract as
    neurst_pt/models/model.py:25-32): `new(args, src_meta, trg_meta)` -> forward / get_symbols_to_logits_fn run through the
    C ABI and agree with the direct implementation."""
    from neurst_b200 import plugin
    from neurst_b200.models import SpeechTransformer, speech_transformer_hparams

    class BaseModel(torch.nn.Module):
        def __init__(self, args):
            self._args = args
            super().__init__()
        args = property(lambda self: self._args)

    cls = plugin._make_model_class(BaseModel, "B200SpeechTransformer", SpeechTransformer, True)
    hp = dict(speech_transformer_hparams("speech_transformer_s")["model.params"])
    hp.update({"modality.source.channels": 64, "modality.dim": 64})
    for side in ("encoder", "decoder"):
        hp.update({side + ".num_layers": 1, side + ".hidden_size": 64, side + ".num_attention_heads": 4, side + ".filter_size": 64})
    src_meta = {"audio_feature_dim": 80, "audio_feature_channels": 1}
    trg_meta = {"vocab_size": 96, "eos_id": 95, "bos_id": 94, "unk_id": 93}
    model = cls.new(hp, src_meta, trg_meta, precision="fp32")
    model.impl.init_parameters(3)
    g = torch.Generator().manual_seed(0)
    inputs = dict(src=torch.randn(2, 50, 80, 1, generator=g), src_length=torch.tensor([50, 33]),
                  trg_input=torch.randint(0, 90, (2, 5), generator=g))
    a = model(inputs, is_training=False)
    direct = SpeechTransformer.new(hp, src_meta, trg_meta, precision="fp32")
    direct.load_parameters({k: v.clone() for k, v in model.named_parameters().items()})
    assert a.shape == (2, 5, 96) and float((a - direct.forward(inputs, is_training=False)).abs().max()) == 0.0
    fn, init = model.get_symbols_to_logits_fn(inputs, is_training=False, is_inference=False)
    assert float((fn(init["decoder_input"], init["decoder_internal_cache"]) - a).abs().max()) == 0.0
