"""CPU tests of the f3 / f4 rows: reference variable names, npz round trip, neurst_pt weight map (against the unmodified
reference module, from the copy oracle/build_ref.py stages), bucket table vs the reference function, SpecAugment sampling rule."""
import os

import numpy as np
import pytest
import torch

from neurst_b200 import checkpoints as CK
from neurst_b200 import data as D
from oracle import build_ref
from oracle import restatement as R

# the reference checkout, or the unmodified copy of it that build() stages under oracle/_ref
REF = os.environ.get("NEURST_REFERENCE") or build_ref.reference_root()
needs_ref = pytest.mark.skipif(not REF, reason="no reference tree and no copy staged by oracle/build_ref.py")


class _FakeRT:
    """Runtime surface used by checkpoints.py, CPU-backed."""

    def __init__(self, cfg, seed=0):
        P = R.init_params(cfg, seed=seed, random_bias=True)
        self.table, off = {}, 0
        for k, v in P.items():
            self.table[k] = (off, tuple(v.shape))
            off += (v.numel() + 7) // 8 * 8
        self.params = torch.zeros(off)
        for k, v in P.items():
            self.view(k).copy_(v)
        self.adam_m = self.adam_v = None
        self._shadow_stale = False

    def view(self, name, arena=None):
        off, shp = self.table[name]
        n = int(np.prod(shp))
        return (self.params if arena is None else arena)[off:off + n].view(*shp)


def test_variable_names_follow_the_reference_scheme():
    cfg = R.CONFIGS["speech_transformer_s"]
    names = CK.tf_variable_names(R.param_shapes(cfg))
    assert len(set(names.values())) == 280
    # SURVEY Appendix B example
    assert names["enc.0.att.qkv.kernel"] == "SpeechTransformer/TransformerEncoder/layer_0/self_attention_prepost_wrapper/self_attention/qkv_transform/kernel"
    assert names["dec.5.cross.kv.bias"] == "SpeechTransformer/TransformerDecoder/layer_5/encdec_attention_prepost_wrapper/encdec_attention/kv_transform/bias"
    assert names["dec.2.ffn.w2"].endswith("layer_2/ffn_prepost_wrapper/ffn/dense2/kernel")
    assert names["enc.3.ffn.ln.gamma"].endswith("layer_3/ffn_prepost_wrapper/ln/gamma")
    assert names["trg.emb"].endswith("target_symbol_modality/shared/weights")


def test_npz_round_trip(tmp_path):
    cfg = R.CONFIGS["speech_transformer_toy"]
    a, b = _FakeRT(cfg, 1), _FakeRT(cfg, 2)
    a.adam_m, a.adam_v = torch.rand_like(a.params), torch.rand_like(a.params)
    p = str(tmp_path / "ckpt.npz")
    CK.save_npz(a, p, scope="MyScope")
    CK.load_npz(b, p)                       # scope auto-detected from the archive
    for k in a.table:
        assert torch.equal(a.view(k), b.view(k)) and torch.equal(a.view(k, a.adam_m), b.view(k, b.adam_m))
    z = np.load(p)
    assert any(n.startswith("MyScope/TransformerEncoder/layer_0/") for n in z.files)
    with pytest.raises(KeyError):
        np.savez(str(tmp_path / "bad.npz"), x=np.zeros(1))
        CK.load_npz(b, str(tmp_path / "bad.npz"))


@needs_ref
def test_weight_map_against_the_unmodified_reference_module():
    """our names -> reference neurst_pt module (to_reference_pt), reference forward == oracle forward on those weights;
    and from_reference_pt inverts it."""
    from oracle import ref_shim
    ref_shim.install()
    from neurst_pt.models import build_model
    from neurst_b200.models import speech_transformer_hparams
    cfg = dict(model="speech", d=16, heads=2, enc_layers=2, dec_layers=2, ffn=24, channels=8, feat=80, in_channels=1, vocab=20)
    hp = dict(speech_transformer_hparams("speech_transformer_s")["model.params"])
    hp.update({"modality.source.channels": 8, "modality.dim": 16})
    for side in ("encoder", "decoder"):
        hp.update({side + ".num_layers": 2, side + ".hidden_size": 16, side + ".num_attention_heads": 2, side + ".filter_size": 24,
                   side + ".attention_dropout_rate": 0.0, side + ".ffn_dropout_rate": 0.0, side + ".layer_postprocess_dropout_rate": 0.0})
    with torch.no_grad():
        model = build_model({"model.class": "SpeechTransformer", "model.params": hp},
                            {"audio_feature_dim": 80, "audio_feature_channels": 1},
                            {"vocab_size": 20, "eos_id": 19, "bos_id": 18, "unk_id": 17})
    P = R.init_params(cfg, seed=5, random_bias=True)
    CK.to_reference_pt(P, model)
    back = CK.from_reference_pt(model)
    assert set(back) == set(P) and all(torch.equal(back[k], P[k]) for k in P)
    g = torch.Generator().manual_seed(0)
    src = torch.randn(2, 41, 80, 1, generator=g)
    lens = torch.tensor([41, 30]); ti = torch.randint(0, 17, (2, 5), generator=g)
    with torch.no_grad():
        ref = model({"src": src, "src_length": lens, "trg_input": ti}, is_training=False)
    mine = R.speech_transformer_forward(P, cfg, src, lens, ti)
    assert float((ref - mine).abs().max()) < 1e-4


def test_bucket_boundaries_match_the_reference_function():
    # the reference function's own outputs (tests/golden/ref_bucket_boundaries.json, oracle/make_golden.py)
    import json
    cases = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_bucket_boundaries.json")))["cases"]
    assert len(cases) == 4
    for c in cases:
        assert D.create_audio_bucket_boundaries(c["maxlen"], c["minlen"]) == c["boundaries"]


def test_frame_budget_bucketer_shapes_and_batches():
    bk = D.FrameBudgetBucketer(24000, 3000, 150, min_src_bucket_boundary=300, world=2, frame_transcript_ratio=12)
    shapes = bk.shapes()
    assert shapes[-1][0] == D.minimal_multiple(3001, 8) and all(b % 8 == 0 and l % 8 == 0 for _, b, l in shapes)
    assert all(t * b <= 24000 + 8 * t for t, b, _ in shapes)
    g = torch.Generator().manual_seed(0)
    ex = [dict(audio=torch.randn(int(n), 80, generator=g), transcript=torch.randint(4, 50, (max(2, int(n) // 40),), generator=g))
          for n in torch.randint(100, 700, (400,), generator=g)]
    got = list(bk.batches(ex))
    assert got, "no batch was formed"
    for per_rank in got:
        assert len(per_rank) == 2 and per_rank[0]["src"].shape == per_rank[1]["src"].shape      # same bucket on every replica
        b = per_rank[0]
        assert int(b["src_length"].max()) <= b["src"].shape[1] and float(b["src"][0, int(b["src_length"][0]):].abs().sum()) == 0.0


def test_specaugment_masks_follow_the_reference_rule():
    sa = D.SpecAugment.build("LD")
    g = torch.Generator().manual_seed(3)
    src = torch.randn(3, 400, 80, 1, generator=g)
    lens = torch.tensor([400, 250, 90])       # 90 < time_mask_t = 100: no time mask for that utterance (audio_lib.py:133-134)
    src[1, 250:] = 0; src[2, 90:] = 0
    out = sa(src, lens, generator=torch.Generator().manual_seed(7))
    changed = (out != src)[..., 0]
    assert changed.any() and not changed[1, 250:].any() and not changed[2, 90:].any()     # padding untouched
    t_rows = changed.all(-1)                                                             # fully masked frames = time masks
    assert not t_rows[2].any()
    assert int(t_rows[0].sum()) <= 2 * 100 and int(changed.any(1)[0].sum()) <= 80
    mean0 = float(src[0, :, :, 0].mean())
    assert abs(float(out[0][changed[0]].mean()) - mean0) < 1e-5                            # filled with the utterance mean


def test_staged_reference_copy_is_unmodified_and_runs():
    """oracle/_ref (oracle/build_ref.py): every staged file is byte-identical to the reference's, and the staged tree —
    the one that travels to the GPU box for bench.py's `cpu_baseline.reference_forward` — reproduces the oracle forward."""
    import hashlib
    import json
    import subprocess
    import sys
    from oracle import build_ref
    root = build_ref.build()
    if root is None:
        pytest.skip("no staged reference and no /root/reference")
    man = json.load(open(os.path.join(root, "MANIFEST.json")))["files"]
    assert len(man) > 20 and "neurst_pt/models/speech_transformer.py" in man
    for rel, digest in man.items():
        assert hashlib.sha256(open(os.path.join(root, rel), "rb").read()).hexdigest() == digest
        if os.path.isdir(os.path.join(build_ref.SRC, "neurst_pt")):
            assert hashlib.sha256(open(os.path.join(build_ref.SRC, rel), "rb").read()).hexdigest() == digest, rel
    code = r'''
import os, sys, torch
sys.path.insert(0, %r)
os.environ["NEURST_REFERENCE_SRC"] = "/nonexistent"          # force the staged tree
from oracle import build_ref, restatement as R
from neurst_b200 import checkpoints as CK
cfg = dict(model="speech", d=16, heads=2, enc_layers=2, dec_layers=2, ffn=24, channels=8, feat=80, in_channels=1, vocab=20)
import importlib; importlib.reload(build_ref)
model = build_ref.reference_speech_transformer(cfg, 20)
import neurst_pt
assert os.path.realpath(neurst_pt.__file__).startswith(os.path.realpath(build_ref.DEST)), neurst_pt.__file__
P = R.init_params(cfg, seed=5, random_bias=True)
CK.to_reference_pt(P, model)
g = torch.Generator().manual_seed(0)
src = torch.randn(2, 41, 80, 1, generator=g); lens = torch.tensor([41, 30]); ti = torch.randint(0, 17, (2, 5), generator=g)
with torch.no_grad():
    ref = model({"src": src, "src_length": lens, "trg_input": ti}, is_training=False)
mine = R.speech_transformer_forward(P, cfg, src, lens, ti)
print("MAXDIFF", float((ref - mine).abs().max()))
''' % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))),)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    diff = float(out.stdout.strip().split("MAXDIFF")[-1])
    assert diff < 1e-4, diff


def test_prefetcher_order_errors_and_shutdown():
    import threading
    seen = []
    p = D.Prefetcher(iter(range(20)), depth=2, init=lambda: seen.append(threading.current_thread().name))
    assert list(p) == list(range(20)) and len(seen) == 1 and seen[0] != threading.current_thread().name

    def bad():
        yield 1
        raise ValueError("boom")
    q = D.Prefetcher(bad())
    assert next(q) == 1
    with pytest.raises(ValueError):
        next(q)

    def endless():
        i = 0
        while True:
            yield torch.full((4,), float(i))
            i += 1
    r = D.Prefetcher(endless(), depth=3)
    assert [float(next(r)[0]) for _ in range(5)] == [0.0, 1.0, 2.0, 3.0, 4.0]
    r.close()
    assert not r._t.is_alive()
