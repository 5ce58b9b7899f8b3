"""ORACLE (test infrastructure only): recipe that stages the UNMODIFIED reference PyTorch mirror for the GPU box.

    python oracle/build_ref.py          # run in the build container (needs /root/reference); also run by __graft_entry__.build()

The reference's only implementation of this path that can run without TensorFlow is `neurst_pt` (forward only: its
autograd fails, SURVEY.md 8c).  It is Python, so "building" it means staging: this script copies
    /root/reference/neurst_pt/**.py           (the models / layers themselves)
    /root/reference/neurst/utils/*.py         (registry, flags, configurable ... imported by neurst_pt)
byte for byte into oracle/_ref/ (git-ignored: reference sources never enter the history; NOT gpurun-ignored: the copy
travels to the GPU box like a built .so) and writes oracle/_ref/MANIFEST.json with the SHA-256 of every file.  Users:
`bench.py`'s CPU legs (`cpu_baseline.reference_forward`, kind "reference": the unmodified reference forward timed on the
host cores) and tests/test_oracle.py (the staged copy reproduces the committed refpt fixtures).  Loaded through
oracle/ref_shim.py with NEURST_REFERENCE pointing at oracle/_ref.
"""
import hashlib
import json
import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")
SRC = os.environ.get("NEURST_REFERENCE_SRC", "/root/reference")


def staged():
    """Path of the staged tree when it is complete, else None."""
    return DEST if os.path.exists(os.path.join(DEST, "MANIFEST.json")) and os.path.isdir(os.path.join(DEST, "neurst_pt")) else None


def build(force=False):
    if not os.path.isdir(os.path.join(SRC, "neurst_pt")):
        return staged()               # GPU box: use what travelled
    files = []
    for sub, recursive in (("neurst_pt", True), (os.path.join("neurst", "utils"), False)):
        root = os.path.join(SRC, sub)
        for d, _, names in os.walk(root):
            for n in sorted(names):
                if n.endswith(".py"):
                    files.append(os.path.relpath(os.path.join(d, n), SRC))
            if not recursive:
                break
    manifest = {}
    for rel in files:
        with open(os.path.join(SRC, rel), "rb") as f:
            manifest[rel] = hashlib.sha256(f.read()).hexdigest()
    mpath = os.path.join(DEST, "MANIFEST.json")
    if not force and os.path.exists(mpath):
        try:
            if json.load(open(mpath)).get("files") == manifest:
                return DEST
        except Exception:
            pass
    tmp = DEST + ".tmp.%d" % os.getpid()
    shutil.rmtree(tmp, ignore_errors=True)
    for rel in files:
        os.makedirs(os.path.dirname(os.path.join(tmp, rel)), exist_ok=True)
        shutil.copyfile(os.path.join(SRC, rel), os.path.join(tmp, rel))
    with open(os.path.join(tmp, "MANIFEST.json"), "w") as f:
        json.dump({"source": "bytedance/neurst (unmodified files, staged by oracle/build_ref.py)", "files": manifest}, f, indent=1)
    shutil.rmtree(DEST, ignore_errors=True)
    os.replace(tmp, DEST)
    return DEST


def reference_root():
    """The reference tree the oracle loads: the source checkout when present, else the copy staged here (None if neither)."""
    return SRC if os.path.isdir(os.path.join(SRC, "neurst_pt")) else staged()


def reference_speech_transformer(hparams, vocab, seed=1234):
    """Instantiates the unmodified reference `neurst_pt` SpeechTransformer (random init) from the staged tree."""
    root = staged() or reference_root()
    if root is None:
        raise RuntimeError("no reference tree: run oracle/build_ref.py in the build container")
    os.environ["NEURST_REFERENCE"] = root
    import importlib
    import torch
    from oracle import ref_shim
    importlib.reload(ref_shim)
    ref_shim.install()
    from neurst_pt.models.speech_transformer import SpeechTransformer
    d = hparams["d"]
    params = {"modality.source.kernel_size": 3, "modality.source.strides": 2, "modality.source.channels": hparams["channels"],
              "modality.source.layer_norm": True, "modality.dim": d, "modality.source.dim": None, "modality.target.dim": None,
              "modality.share_embedding_and_softmax_weights": True, "modality.timing": "sinusoids",
              "modality.source.timing": None, "modality.target.timing": None}
    for side, nl in (("encoder", hparams["enc_layers"]), ("decoder", hparams["dec_layers"])):
        params.update({side + ".num_layers": nl, side + ".hidden_size": d, side + ".num_attention_heads": hparams["heads"],
                       side + ".filter_size": hparams["ffn"], side + ".attention_dropout_rate": 0.1, side + ".attention_type": "dot_product",
                       side + ".ffn_activation": "relu", side + ".ffn_dropout_rate": 0.1, side + ".layer_postprocess_dropout_rate": 0.1,
                       side + ".layer_postprocess_epsilon": 1e-6})
    torch.manual_seed(seed)
    with torch.no_grad():
        return SpeechTransformer.new(params, {"audio_feature_dim": 80, "audio_feature_channels": 1},
                                     {"vocab_size": vocab, "eos_id": vocab - 1, "bos_id": vocab - 2, "unk_id": vocab - 3})


if __name__ == "__main__":
    print(build(force=True))
