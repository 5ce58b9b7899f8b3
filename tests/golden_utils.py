"""Helpers shared by the oracle (CPU) and CUDA-parity (GPU) tests: load the committed golden fixtures and
map the reference's TF variable names onto the flat parameter names used by oracle/ and neurst_b200/."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz")))


def t(a, dtype=torch.float32):
    return torch.tensor(np.asarray(a), dtype=dtype)


_TF_SUB = [
    ("self_attention_prepost_wrapper/self_attention/output_transform/kernel", "{}.out.kernel", "att"),
    ("self_attention_prepost_wrapper/self_attention/qkv_transform/kernel", "{}.qkv.kernel", "att"),
    ("encdec_attention_prepost_wrapper/encdec_attention/output_transform/kernel", "{}.out.kernel", "cross"),
    ("encdec_attention_prepost_wrapper/encdec_attention/q_transform/kernel", "{}.q.kernel", "cross"),
    ("encdec_attention_prepost_wrapper/encdec_attention/kv_transform/kernel", "{}.kv.kernel", "cross"),
    ("ffn_prepost_wrapper/ffn/dense1/kernel", "{}.w1", "ffn"),
    ("ffn_prepost_wrapper/ffn/dense2/kernel", "{}.w2", "ffn"),
]


def tf_name_to_flat(name, default_stack):
    """'TransformerEncoder/layer_0/ffn_prepost_wrapper/ffn/dense1/kernel' -> 'enc.0.ffn.w1'."""
    stack = default_stack
    if "TransformerEncoder" in name:
        stack = "enc"
    elif "TransformerDecoder" in name:
        stack = "dec"
    layer = int(name.split("layer_")[1].split("/")[0])
    for sub, fmt, kind in _TF_SUB:
        if sub in name:
            if kind == "att":
                kind = "att" if stack == "enc" else "self"
            return fmt.format("%s.%d.%s" % (stack, layer, kind))
    raise KeyError(name)


def default_params(cfg, dtype=torch.float32):
    """Reference defaults for everything a KAT does not assign: zero biases, LN gamma=1 / beta=0."""
    from oracle import restatement as R
    P = {}
    for name, shp in R.param_shapes(cfg).items():
        P[name] = torch.ones(shp, dtype=dtype) if name.endswith(".gamma") else torch.zeros(shp, dtype=dtype)
    return P


def kat_params(kat, cfg, default_stack, dtype=torch.float32):
    P = default_params(cfg, dtype)
    for k, v in kat.items():
        if k.startswith("w:") and "layer_" in k:
            P[tf_name_to_flat(k[2:], default_stack)] = t(v, dtype)
    return P


def refpt_case(name, dtype=torch.float32):
    """Fixture, weights and config of a refpt_* case.  The fixture stores the weight seed: the reference ran on
    oracle.restatement.init_params(cfg, seed, random_bias=True), regenerated here bit for bit."""
    from oracle import restatement as R
    z = load(name)
    d, heads, enc_layers, dec_layers, ffn, channels, vocab = [int(x) for x in z["cfg"]]
    cfg = dict(model="speech", d=d, heads=heads, enc_layers=enc_layers, dec_layers=dec_layers, ffn=ffn,
               channels=channels, feat=80, in_channels=1, vocab=vocab)
    P = {k: v.to(dtype) for k, v in R.init_params(cfg, seed=int(z["seed"]), random_bias=True).items()}
    return z, P, cfg
