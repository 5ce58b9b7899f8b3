"""ORACLE (test infrastructure only): generates the reference-derived fixtures under tests/golden/
(`NEURST_REFERENCE=<reference checkout> python oracle/make_golden.py`).  The tests read only what it wrote, never the
reference itself.

Three kinds of fixtures:
  kat_*.npz   — the TF-generated known-answer vectors hard-coded in the reference's own tests
                (tests/neurst/**), extracted here by parsing those test files' literals with `ast`
                (weights, inputs, expected outputs; nothing is executed).
  refpt_*.npz — inputs, weight seed and outputs of the UNMODIFIED reference PyTorch mirror (neurst_pt) run on CPU
                through oracle/ref_shim.py.
  ref_bucket_boundaries.json — the reference's length-bucket table at a few arguments.
"""
import ast
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = os.environ.get("NEURST_REFERENCE", "/root/reference")
OUT = os.path.join(ROOT, "tests", "golden")


# ----------------------------------------------------------------------------------------------
# KAT extraction
# ----------------------------------------------------------------------------------------------
def _num_literal(node):
    """Returns a numpy array if `node` (or its first positional arg, for tf.convert_to_tensor / numpy.array
    calls) is a nested numeric list literal, else None."""
    if isinstance(node, ast.Call) and node.args:
        return _num_literal(node.args[0])
    if isinstance(node, (ast.List, ast.Tuple)):
        try:
            return np.array(ast.literal_eval(node), dtype=np.float64)
        except Exception:
            return None
    return None


def _first_literal(nodes):
    for n in nodes:
        for sub in ast.walk(n):
            if isinstance(sub, ast.Call):
                arr = _num_literal(sub)
                if arr is not None and arr.size > 0:
                    return arr
    return None


def _str_consts(node):
    return [s.value for s in ast.walk(node) if isinstance(s, ast.Constant) and isinstance(s.value, str)]


def extract_kat(path, func):
    """dict with keys  w:<substring tested against w.name>  |  shape:<tuple>  |  var:<assigned name>  |
    dict:<key> (literal dict entries)  |  expect:<i> (literals inside assert statements, in order)."""
    tree = ast.parse(open(path).read())
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == func][0]
    out = {}
    n_expect = 0

    def visit_if(node):
        test = node.test
        key = None
        strs = _str_consts(test)
        if strs:
            key = "w:" + "".join(strs)
        elif isinstance(test, ast.Compare) and isinstance(test.comparators[0], ast.Tuple):
            key = "shape:" + str(tuple(ast.literal_eval(test.comparators[0])))
        arr = _first_literal(node.body)
        if key is not None and arr is not None:
            out[key] = arr
        for o in node.orelse:
            if isinstance(o, ast.If):
                visit_if(o)

    for node in ast.walk(fn):
        if isinstance(node, ast.Assign) and len(node.targets) == 1 and isinstance(node.targets[0], ast.Name):
            arr = _num_literal(node.value) if isinstance(node.value, (ast.Call, ast.List)) else None
            if arr is not None and arr.size > 0:
                out.setdefault("var:" + node.targets[0].id, arr)
            if isinstance(node.value, ast.Dict):
                for k, v in zip(node.value.keys, node.value.values):
                    a = _num_literal(v)
                    if a is not None and isinstance(k, ast.Constant):
                        out["dict:" + str(k.value)] = a
    for node in fn.body:
        for sub in ast.walk(node):
            if isinstance(sub, ast.If):
                visit_if(sub)
            if (isinstance(sub, ast.Call) and isinstance(sub.func, ast.Attribute) and sub.func.attr == "set_weights"
                    and "call:set_weights" not in out):
                arr = _first_literal(sub.args)
                if arr is not None:
                    out["call:set_weights"] = arr
    for node in ast.walk(fn):
        if isinstance(node, ast.Assert) or (isinstance(node, ast.Expr) and isinstance(node.value, ast.Call)
                                            and "assert" in ast.dump(node.value.func)):
            for sub in ast.walk(node):
                if isinstance(sub, ast.Call):
                    a = _num_literal(sub)
                    if a is not None and a.size > 1 and isinstance(sub.func, ast.Attribute) and sub.func.attr == "array":
                        out["expect:%d" % n_expect] = a
                        n_expect += 1
    return out


KATS = [
    ("kat_mha_cross", "tests/neurst/layers/attentions/multi_head_attention_test.py", "test_multihead_attention"),
    ("kat_mha_self", "tests/neurst/layers/attentions/multi_head_attention_test.py", "test_multiheadself_attention"),
    ("kat_mha_self_cache", "tests/neurst/layers/attentions/multi_head_attention_test.py",
     "test_multiheadself_attention_under_dec"),
    ("kat_encoder", "tests/neurst/layers/encoders/transformer_encoder_test.py", "test_transformer_encoder"),
    ("kat_decoder", "tests/neurst/layers/decoders/transformer_decoder_test.py", "test_transformer_decoder"),
    ("kat_transformer", "tests/neurst/models/transformer_test.py", "test_seq2seq"),
    ("kat_position", "tests/neurst/layers/common_layers_test.py", "test_position_embedding"),
]


def make_kats():
    for name, rel, func in KATS:
        path = os.path.join(REF, rel)
        try:
            d = extract_kat(path, func)
        except IndexError:
            print("skip %s: %s not found" % (name, func))
            continue
        np.savez(os.path.join(OUT, name + ".npz"), **d)
        print(name, {k: v.shape for k, v in d.items()})


# ----------------------------------------------------------------------------------------------
# reference-PT generated fixtures
# ----------------------------------------------------------------------------------------------
def make_refpt():
    """Weights are `restatement.init_params(cfg, seed, random_bias=True)`, copied into the reference module through
    neurst_b200.checkpoints.to_reference_pt; the fixture stores the seed instead of the weights (tests/golden_utils.py
    regenerates them), which keeps it small and pins the weight map along with the forward."""
    import torch
    from oracle import ref_shim
    from oracle import restatement as R
    from neurst_b200 import checkpoints as CK
    ref_shim.install()
    from neurst_pt.models.speech_transformer import SpeechTransformer

    def build(d, heads, enc_layers, dec_layers, ffn_size, channels, vocab, seed):
        params = {
            "modality.source.kernel_size": 3, "modality.source.strides": 2, "modality.source.channels": channels,
            "modality.source.layer_norm": True, "modality.dim": d, "modality.source.dim": None,
            "modality.target.dim": None, "modality.share_embedding_and_softmax_weights": True,
            "modality.timing": "sinusoids", "modality.source.timing": None, "modality.target.timing": None,
        }
        for side, nl in (("encoder", enc_layers), ("decoder", dec_layers)):
            params.update({side + ".num_layers": nl, side + ".hidden_size": d, side + ".num_attention_heads": heads,
                           side + ".filter_size": ffn_size, side + ".attention_dropout_rate": 0.1,
                           side + ".attention_type": "dot_product", side + ".ffn_activation": "relu",
                           side + ".ffn_dropout_rate": 0.1, side + ".layer_postprocess_dropout_rate": 0.1,
                           side + ".layer_postprocess_epsilon": 1e-6})
        src_meta = {"audio_feature_dim": 80, "audio_feature_channels": 1}
        trg_meta = {"vocab_size": vocab, "eos_id": vocab - 1, "bos_id": vocab - 2, "unk_id": vocab - 3}
        cfg = dict(model="speech", d=d, heads=heads, enc_layers=enc_layers, dec_layers=dec_layers, ffn=ffn_size,
                   channels=channels, feat=80, in_channels=1, vocab=vocab)
        P = R.init_params(cfg, seed=seed, random_bias=True)
        with torch.no_grad():
            model = SpeechTransformer.new(params, src_meta, trg_meta)
            CK.to_reference_pt(P, model)
        back = CK.from_reference_pt(model)
        assert set(back) == set(P) and all(torch.equal(back[k], P[k]) for k in P)
        return model

    cases = [
        ("refpt_speech_toy", dict(d=8, heads=2, enc_layers=2, dec_layers=2, ffn_size=10, channels=5, vocab=12, seed=11),
         dict(B=3, T=37, L=5, lengths=[37, 30, 18])),
        ("refpt_speech_small", dict(d=64, heads=4, enc_layers=2, dec_layers=2, ffn_size=128, channels=64, vocab=96, seed=12),
         dict(B=2, T=50, L=7, lengths=[50, 41])),
    ]
    for name, mk, io in cases:
        model = build(**mk)
        g = torch.Generator().manual_seed(100 + mk["seed"])
        B, T, L = io["B"], io["T"], io["L"]
        src = torch.randn(B, T, 80, 1, generator=g)
        lengths = torch.tensor(io["lengths"], dtype=torch.long)
        for b in range(B):
            src[b, io["lengths"][b]:] = 0.0
        trg_input = torch.randint(0, mk["vocab"], (B, L), generator=g)
        with torch.no_grad():
            logits = model({"src": src.clone(), "src_length": lengths, "trg_input": trg_input}, is_training=False)
            sm = model._src_modality
            emb = sm(src.clone())
            conv = sm._embedding_layer(src.clone())
        np.savez(os.path.join(OUT, name + ".npz"), src=src.numpy(), src_length=lengths.numpy(),
                 trg_input=trg_input.numpy(), logits=logits.numpy(), emb=emb.numpy(), conv=conv.numpy(),
                 cfg=np.array([mk["d"], mk["heads"], mk["enc_layers"], mk["dec_layers"], mk["ffn_size"], mk["channels"],
                               mk["vocab"]]), seed=np.array(mk["seed"]))
        print(name, "logits", tuple(logits.shape))


# ----------------------------------------------------------------------------------------------
# reference functions evaluated at fixed arguments
# ----------------------------------------------------------------------------------------------
BUCKET_ARGS = [(3000, 128), (2000, 100), (800, None), (3000, 300)]


def make_bucket_boundaries():
    """neurst/tasks/speech2text.py `create_audio_bucket_boundaries`, loaded from the source with `ast` (the module itself
    imports TensorFlow) and evaluated at BUCKET_ARGS."""
    import json
    import math
    src = open(os.path.join(REF, "neurst/tasks/speech2text.py")).read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "create_audio_bucket_boundaries")
    ns = {"math": math}
    exec(compile(ast.Module([fn], []), "ref", "exec"), ns)
    cases = [{"maxlen": a, "minlen": b, "boundaries": ns["create_audio_bucket_boundaries"](a, b)} for a, b in BUCKET_ARGS]
    with open(os.path.join(OUT, "ref_bucket_boundaries.json"), "w") as f:
        json.dump({"source": "reference neurst/tasks/speech2text.py create_audio_bucket_boundaries", "cases": cases}, f, indent=1)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    make_kats()
    make_refpt()
    make_bucket_boundaries()
