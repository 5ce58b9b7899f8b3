"""Generates tests/golden/tfrecord_fixture.json from the reference's own TFRecord fixtures
(/root/reference/tests/examples/train.tfrecords-0000?-of-00004, written by TensorFlow from train.example.*.bpe.txt with
tests/examples/example_create_seq2seq_tfrecrods.yml).  Run in the build container (the GPU box has no /root/reference):

    python tests/golden/make_tfrecord_fixture.py

Stored: per file the record count and a SHA-256 over the record payloads; the first two framed records of shard 0 verbatim
(hex, 16 framing bytes + payload each) with the ids an INDEPENDENT decoder (the google.protobuf runtime on a descriptor
built from the published example.proto / feature.proto) reads from them, and the text those ids spell in the reference's
vocabulary (vocab.en) — which is line 4 / line 5 of train.example.en.tok.bpe.txt, the text the records were made from.
Beside the JSON, a sample of the fixture itself: shard 0 and vocab.en gzipped, and a 64-bit digest of every line of
train.example.en.tok.bpe.txt (line_digest) in place of the text.
"""
import glob
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
EX = "/root/reference/tests/examples"


def example_class():
    """tf.train.Example rebuilt on the protobuf runtime (schema of tensorflow/core/example/{feature,example}.proto)."""
    from google.protobuf import descriptor_pb2, descriptor_pool, message_factory
    fd = descriptor_pb2.FileDescriptorProto(name="b200st_example.proto", package="b200st_tf", syntax="proto3")
    T = descriptor_pb2.FieldDescriptorProto

    def msg(name, fields):
        m = fd.message_type.add(name=name)
        for fname, num, typ, label, tname, packed in fields:
            f = m.field.add(name=fname, number=num, type=typ, label=label)
            if tname:
                f.type_name = tname
            if packed is not None:
                f.options.packed = packed
        return m
    msg("BytesList", [("value", 1, T.TYPE_BYTES, T.LABEL_REPEATED, None, None)])
    msg("FloatList", [("value", 1, T.TYPE_FLOAT, T.LABEL_REPEATED, None, True)])
    msg("Int64List", [("value", 1, T.TYPE_INT64, T.LABEL_REPEATED, None, True)])
    feat = msg("Feature", [("bytes_list", 1, T.TYPE_MESSAGE, T.LABEL_OPTIONAL, ".b200st_tf.BytesList", None),
                           ("float_list", 2, T.TYPE_MESSAGE, T.LABEL_OPTIONAL, ".b200st_tf.FloatList", None),
                           ("int64_list", 3, T.TYPE_MESSAGE, T.LABEL_OPTIONAL, ".b200st_tf.Int64List", None)])
    feat.oneof_decl.add(name="kind")
    for f in feat.field:
        f.oneof_index = 0
    feats = msg("Features", [("feature", 1, T.TYPE_MESSAGE, T.LABEL_REPEATED, ".b200st_tf.Features.FeatureEntry", None)])
    entry = feats.nested_type.add(name="FeatureEntry")
    entry.options.map_entry = True
    entry.field.add(name="key", number=1, type=T.TYPE_STRING, label=T.LABEL_OPTIONAL)
    entry.field.add(name="value", number=2, type=T.TYPE_MESSAGE, label=T.LABEL_OPTIONAL, type_name=".b200st_tf.Feature")
    msg("Example", [("features", 1, T.TYPE_MESSAGE, T.LABEL_OPTIONAL, ".b200st_tf.Features", None)])
    pool = descriptor_pool.DescriptorPool()
    pool.Add(fd)
    return message_factory.GetMessageClass(pool.FindMessageTypeByName("b200st_tf.Example"))


def line_digest(text):
    """First 8 bytes of the SHA-256 of a UTF-8 line, as an unsigned little-endian integer."""
    return int.from_bytes(hashlib.sha256(text.encode("utf-8")).digest()[:8], "little")


def write_samples(lines):
    import gzip
    import numpy as np
    gold = os.path.join(ROOT, "tests", "golden")
    shard0 = sorted(glob.glob(os.path.join(EX, "train.tfrecords-*")))[0]
    for src, dst in ((shard0, "ref_" + os.path.basename(shard0) + ".gz"), (os.path.join(EX, "vocab.en"), "ref_vocab.en.gz")):
        with open(src, "rb") as fi, gzip.GzipFile(os.path.join(gold, dst), "wb", mtime=0) as fo:
            fo.write(fi.read())
    np.save(os.path.join(gold, "ref_train_en_line_digests.npy"), np.array(sorted(line_digest(l) for l in lines), np.uint64))


def main():
    import numpy as np
    from neurst_b200 import tfrecord as R
    Example = example_class()
    vocab = [l.rstrip("\n").split("\t")[0].split(" ")[0] for l in open(os.path.join(EX, "vocab.en"), encoding="utf-8")]
    lines = [l.rstrip("\n") for l in open(os.path.join(EX, "train.example.en.tok.bpe.txt"), encoding="utf-8")]
    out = {"source": "reference tests/examples/train.tfrecords-0000?-of-00004 (TensorFlow-written)", "files": [], "records": []}
    for f in sorted(glob.glob(os.path.join(EX, "train.tfrecords-*"))):
        h = hashlib.sha256()
        n = labels = 0
        for rec in R.read_records(f, verify=2):
            h.update(rec.tobytes())
            n += 1
        out["files"].append({"name": os.path.basename(f), "records": n, "payload_sha256": h.hexdigest()})
    f0 = sorted(glob.glob(os.path.join(EX, "train.tfrecords-*")))[0]
    img = np.fromfile(f0, np.uint8)
    pos = 0
    for _ in range(2):
        ln = int(img[pos:pos + 8].view("<u8")[0])
        framed = img[pos:pos + 16 + ln]
        ex = Example.FromString(img[pos + 12:pos + 12 + ln].tobytes())
        ids = {k: [int(x) for x in v.int64_list.value] for k, v in ex.features.feature.items()}
        text = " ".join(vocab[i] for i in ids["label"] if i < len(vocab))
        out["records"].append({"framed_hex": framed.tobytes().hex(), "ids": ids, "label_text": text,
                               "label_text_line": lines.index(text)})
        pos += 16 + ln
    with open(os.path.join(ROOT, "tests", "golden", "tfrecord_fixture.json"), "w") as fo:
        json.dump(out, fo, indent=1)
    write_samples(lines)
    print(json.dumps(out["files"], indent=1))
    print([(r["label_text_line"], r["label_text"]) for r in out["records"]])


if __name__ == "__main__":
    main()
