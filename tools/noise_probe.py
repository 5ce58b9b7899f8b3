"""Dev tool: run-to-run noise of the gradient arena (same batch, same dropout seed, repeated eager backward passes)
in the default mode, the deterministic mode, without the fused attention / FFN kernels, and at a larger batch."""
import sys
sys.path.insert(0, ".")
import torch
from neurst_b200 import lib as L
from neurst_b200.runtime import Runtime, make_config
from neurst_b200.trainer import synthetic_batch
from oracle import restatement as R

def probe(tag, prec="fp16", dropout=0.1, disable_fused=False, B=4, T=160, Lq=12, deterministic=False):
    cfg = dict(R.CONFIGS["speech_transformer_s"]); cfg["vocab"] = 96
    c = make_config(L.MODEL_SPEECH, cfg["d"], cfg["heads"], cfg["ffn"], cfg["enc_layers"], cfg["dec_layers"], 96, channels=256,
                    precision=prec, attention_dropout=dropout, ffn_dropout=dropout, postprocess_dropout=dropout, label_smoothing=0.1,
                    disable_fused_attention=disable_fused, deterministic=deterministic)
    rt = Runtime(c)
    rt.load_parameters(R.init_params(cfg, seed=5))
    batch = synthetic_batch(B, T, Lq, 96, seed=100, device="cuda")
    b = dict(batch); b.update(training=dropout > 0, seed=77, want_logits=True)
    gs, lg = [], []
    for _ in range(3):
        rt.ensure_grads().zero_()
        out = rt.run(b, backward=True)
        torch.cuda.synchronize()
        gs.append(rt.grads.clone()); lg.append(out["logits"].clone())
    n = gs[0].norm()
    print("%-34s grads rel diff %.3e %.3e | logits max diff %.3e" % (tag, float((gs[1] - gs[0]).norm() / n), float((gs[2] - gs[0]).norm() / n),
                                                                    float((lg[1] - lg[0]).abs().max())), flush=True)

probe("fp16 default")
probe("fp16 deterministic slices", deterministic=True)
probe("fp16 no fused attention / FFN", disable_fused=True)
probe("fp16 big batch", B=8, T=400, Lq=40)
