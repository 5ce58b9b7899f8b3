"""Input edge (SURVEY.md 8 f4): TFRecord framing + CRC-32C (libb200st_io, C), tf.train.Example wire format, the
reference's deterministic file interleave / sharding, AudioTFRecordDataset and the SpeechToText batching.

Pins: CRC-32C known answers (RFC 3720 B.4); two records written by TensorFlow, taken verbatim from the reference's own
fixture (tests/golden/tfrecord_fixture.json, made by tests/golden/make_tfrecord_fixture.py), whose ids were read by an
independent decoder (google.protobuf runtime) and spell lines of the text the reference built the records from; the first
shard of that fixture, read whole; the protobuf runtime as a second encoder/decoder of the same schema."""
import gzip
import hashlib
import importlib.util
import json
import os

import numpy as np
import pytest
import torch

from neurst_b200 import data as D
from neurst_b200 import tfrecord as R

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "tfrecord_fixture.json")))


def _fixture_module():
    spec = importlib.util.spec_from_file_location("make_tfrecord_fixture", os.path.join(HERE, "golden", "make_tfrecord_fixture.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _example_class():
    return _fixture_module().example_class()


def test_crc32c_known_answers():
    assert R.crc32c(b"123456789") == 0xE3069283
    assert R.crc32c(bytes(32)) == 0x8A9136AA                       # RFC 3720 B.4
    assert R.crc32c(b"\xff" * 32) == 0x62A8AB43
    assert R.crc32c(bytes(range(32))) == 0x46DD794E
    assert R.crc32c(bytes(range(31, -1, -1))) == 0x113FDB5C
    data = np.random.default_rng(0).integers(0, 256, 100003, dtype=np.uint8).tobytes()
    assert R.crc32c(data[5000:], R.crc32c(data[:5000])) == R.crc32c(data)      # incremental == one shot (unaligned split)


def test_records_written_by_tensorflow(tmp_path):
    raw = b"".join(bytes.fromhex(r["framed_hex"]) for r in GOLD["records"])
    p = tmp_path / "two.tfrecords"
    p.write_bytes(raw)
    recs = list(R.read_records(str(p), verify=2))                   # both CRCs of both records check out
    assert len(recs) == 2
    for rec, g in zip(recs, GOLD["records"]):
        ex = R.parse_example(rec)
        assert set(ex) == set(g["ids"])
        for k, ids in g["ids"].items():
            assert ex[k][0] == "int64" and ex[k][1].tolist() == ids
        assert R.encode_example({k: np.array(v) for k, v in g["ids"].items()}) == rec.tobytes()    # byte-identical re-encoding
    # the writer reproduces TensorFlow's framing bit for bit
    q = tmp_path / "again.tfrecords"
    with R.TFRecordWriter(str(q)) as w:
        for rec in recs:
            w.write(rec.tobytes())
    assert q.read_bytes() == raw
    # damage: payload byte, length byte, truncation -> DataLoss
    for pos in (20, 3):
        bad = bytearray(raw); bad[pos] ^= 0x40
        p.write_bytes(bytes(bad))
        with pytest.raises(R.TFRecordError):
            list(R.read_records(str(p), verify=2))
    p.write_bytes(raw[:-3])
    with pytest.raises(R.TFRecordError):
        list(R.read_records(str(p), verify=0))
    p.write_bytes(b"")
    assert list(R.read_records(str(p))) == []


def test_reference_fixture_first_shard(tmp_path):
    """Shard 0 of the reference's TensorFlow-written fixture (stored gzipped under tests/golden) read end to end."""
    g = GOLD["files"][0]
    with gzip.open(os.path.join(HERE, "golden", "ref_" + g["name"] + ".gz"), "rb") as f:
        (tmp_path / g["name"]).write_bytes(f.read())
    h, n = hashlib.sha256(), 0
    for rec in R.read_records(str(tmp_path / g["name"]), verify=2):
        h.update(rec.tobytes()); n += 1
    assert (n, h.hexdigest()) == (g["records"], g["payload_sha256"])
    # every target decodes, EOS-terminated, to a line of the text the records were built from (stored as line digests:
    # 7594 lines <-> 7594 records over the four shards)
    with gzip.open(os.path.join(HERE, "golden", "ref_vocab.en.gz"), "rt", encoding="utf-8") as f:
        vocab = [l.rstrip("\n").split(" ")[0] for l in f]
    lines = np.load(os.path.join(HERE, "golden", "ref_train_en_line_digests.npy"))
    assert len(lines) == sum(f["records"] for f in GOLD["files"]) == 7594
    line_digest, lines = _fixture_module().line_digest, set(lines.tolist())
    got = []
    for el in R.load_tfrecords(str(tmp_path / "train.tfrecords"), {"feature": R.VarLenInt64, "label": R.VarLenInt64}):
        ids = el["label"]
        assert ids[-1] == len(vocab) + 2                            # EOS id of the reference's vocabulary wrapper
        got.append(" ".join(vocab[i] if i < len(vocab) else "<unk>" for i in ids[:-1]))
    assert len(got) == n
    same = sum(line_digest(t) in lines for t in got)
    assert same > 0.97 * n                                          # the rest contain out-of-vocabulary pieces (<unk>)


def test_example_codec_against_the_protobuf_runtime():
    Example = _example_class()
    rng = np.random.default_rng(1)
    feats = {"audio": rng.standard_normal(57 * 80).astype(np.float32),
             "transcript": np.array([5, 127, 128, 300, 16384, 2 ** 40, -1, -2 ** 63, 2 ** 63 - 1, 0], np.int64),
             "src_lang": "en", "uuid": [b"ted_1_0", b"\xff\x00"], "empty_f": np.empty(0, np.float32), "empty_i": np.empty(0, np.int64)}
    mine = R.encode_example(feats)
    ex = Example.FromString(mine)                                   # the runtime reads what we wrote
    f = ex.features.feature
    assert np.array_equal(np.array(f["audio"].float_list.value, np.float32), feats["audio"])
    assert list(f["transcript"].int64_list.value) == feats["transcript"].tolist()
    assert list(f["src_lang"].bytes_list.value) == [b"en"] and list(f["uuid"].bytes_list.value) == feats["uuid"]
    assert f["empty_f"].WhichOneof("kind") == "float_list" and len(f["empty_f"].float_list.value) == 0
    theirs = ex.SerializeToString(deterministic=True)               # and we read what the runtime writes
    for blob in (mine, theirs):
        got = R.parse_example(blob)
        assert got["audio"][0] == "float" and np.array_equal(got["audio"][1], feats["audio"])
        assert got["transcript"][0] == "int64" and np.array_equal(got["transcript"][1], feats["transcript"])
        assert got["uuid"] == ("bytes", feats["uuid"]) and got["src_lang"] == ("bytes", [b"en"])
        assert got["empty_f"][1].size == 0 and got["empty_i"][1].size == 0
    assert mine == theirs                                           # same bytes as the deterministic C++/upb serializer
    # unpacked repeated scalars (older writers) are accepted too
    unpacked = R._ld(1, R._ld(1, R._ld(1, b"x") + R._ld(2, R._ld(3, b"\x08\x07\x08\x81\x01") + b"")))
    assert R.parse_example(unpacked)["x"][1].tolist() == [7, 129]
    with pytest.raises(R.TFRecordError):
        R.parse_example(mine[:-2])


def _write(path, values):
    with R.TFRecordWriter(str(path)) as w:
        for v in values:
            w.write(R.encode_example({"id": np.array([v])}))


def test_interleave_order_and_file_sharding(tmp_path):
    counts = {"train-00000": 3, "train-00001": 1, "train-00002": 2, "train-00003": 0, "train-00004": 2}
    for k, (name, n) in enumerate(sorted(counts.items())):
        _write(tmp_path / name, [100 * k + j for j in range(n)])
    ids = lambda **kw: [int(e["id"][0]) for e in R.load_tfrecords(str(tmp_path), {"id": R.VarLenInt64}, **kw)]
    # Dataset.interleave(cycle_length=2, block_length=1): A0 B0 A1 | B ends -> C takes its slot: C0 A2 C1 | A ends -> D (empty) -> E
    assert ids(cycle_length=2) == [0, 100, 1, 200, 2, 201, 400, 401]
    assert ids() == [0, 100, 200, 400, 1, 201, 401, 2]                                   # cycle_length 10: plain round robin
    assert ids(num_shards=2, sharding_index=0) == [0, 200, 400, 1, 201, 401, 2]           # files 0, 2, 4
    assert ids(num_shards=2, sharding_index=1) == [100]                                   # files 1, 3
    assert R.glob_tfrecords(str(tmp_path / "train-0000")) == sorted(str(tmp_path / n) for n in counts)   # prefix -> prefix*
    assert R.glob_tfrecords([str(tmp_path / "train-00001"), str(tmp_path / "train-00004")]) == [
        str(tmp_path / "train-00001"), str(tmp_path / "train-00004")]


def _audio_records(path, n, rng, projected=True):
    lens = []
    with R.TFRecordWriter(str(path)) as w:
        for i in range(n):
            frames = int(rng.integers(90, 640))
            l = max(2, frames // 30)
            lens.append((frames, l))
            tr = np.concatenate([rng.integers(4, 90, l - 1), [2]]) if projected else "hello world %d" % i
            w.write(R.encode_example({"audio": rng.standard_normal(frames * 80).astype(np.float32), "transcript": tr,
                                      "src_lang": "en", "uuid": "utt_%d" % i}))
    return lens


def test_audio_tfrecord_dataset_and_speech_to_text_batches(tmp_path):
    rng = np.random.default_rng(5)
    lens = []
    for s in range(3):
        lens.append(_audio_records(tmp_path / ("train.tfrecords-%05d-of-00003" % s), 150, rng))
    ds = R.AudioTFRecordDataset({"data_path": str(tmp_path / "train.tfrecords")})
    assert ds.status == {"audio": "projected", "transcript": "projected"}
    assert ds.fields == {"audio": "float", "transcript": "int64", "src_lang": "bytes", "uuid": "bytes"}
    first = next(ds.build_iterator()())
    assert first["uuid"] == "utt_0" and first["src_lang"] == "en" and first["audio"].shape == (lens[0][0][0] * 80,)
    assert [e["uuid"] for e in ds.build_iterator(shard_id=1, total_shards=3)()][:2] == ["utt_0", "utt_1"]     # file 1 only
    assert sum(1 for _ in ds.build_iterator(shard_id=1, total_shards=3)()) == 150

    task = D.SpeechToText({"pad_id": 0, "bos_id": 1, "eos_id": 2}, max_src_len=600, max_trg_len=24, batch_size_per_gpu=4000,
                          min_src_bucket_boundary=128, frame_transcript_ratio=30, world=2)
    proc = task.preprocess_fn(ds.status)
    steps = list(task.train_batches(ds.build_iterator(map_func=proc)()))
    assert steps
    shapes = set(task.bucketer.shapes())
    seen = 0
    for per_rank in steps:
        assert len(per_rank) == 2
        a, b = per_rank
        assert a["src"].shape == b["src"].shape and a["trg"].shape == b["trg"].shape
        B, T, L = a["src"].shape[0], a["src"].shape[1], a["trg"].shape[1]
        assert (T, B, L) in shapes and a["src"].shape[2:] == (80, 1)
        for d in per_rank:
            seen += B
            assert int(d["src_length"].max()) <= T and int(d["src_length"].min()) > 0
            assert torch.equal(d["trg_input"][:, 0], torch.ones(B, dtype=torch.long)) and torch.equal(d["trg_input"][:, 1:], d["trg"][:, :-1])
            assert torch.equal(d["trg_length"], (d["trg"] != 0).sum(1))
            j = int(d["trg_length"][0])
            assert int(d["trg"][0, j - 1]) == 2 and float(d["src"][0, int(d["src_length"][0]):].abs().sum()) == 0.0
    kept = sum(1 for fl in lens for (f, l) in fl if f <= 600 and 1 < l <= 24)
    assert 0 < seen <= kept                                          # the remainder of every bucket is dropped (drop_remainder)

    # a transcript too long for its own audio bucket's two bounds moves to the first later bucket that takes it
    bk = task.bucketer
    i0, _ = bk.bucket_of(100, 2)
    long_t = bk.trg_pairs[i0][1] + 1
    moved = bk.bucket_of(100, long_t)
    assert moved is not None and moved[0] > i0 and long_t <= bk.trg_pairs[moved[0]][moved[1]]
    assert bk.bucket_of(601 + 8, 2) is None

    # raw text is refused with the reason
    _audio_records(tmp_path / "raw.tfrecords", 3, rng, projected=False)
    raw = R.AudioTFRecordDataset({"data_path": str(tmp_path / "raw.tfrecords")})
    assert raw.status["transcript"] == "raw" and next(raw.build_iterator()())["transcript"] == "hello world 0"
    with pytest.raises(RuntimeError):
        task.preprocess_fn(raw.status)



def test_specaugment_in_batches_is_reproducible(tmp_path):
    rng = np.random.default_rng(9)
    _audio_records(tmp_path / "train.tfrecords-00000-of-00001", 200, rng)
    ds = R.AudioTFRecordDataset({"data_path": str(tmp_path / "train.tfrecords")})

    def run(seed):
        task = D.SpeechToText({"pad_id": 0, "bos_id": 1, "eos_id": 2}, max_src_len=640, max_trg_len=24, batch_size_per_gpu=4000,
                              frame_transcript_ratio=30, specaug="SM")
        g = torch.Generator().manual_seed(seed)
        return list(task.train_batches(ds.build_iterator(map_func=task.preprocess_fn(ds.status))(), generator=g))
    a, b, c = run(4), run(4), run(5)
    assert len(a) == len(b) == len(c) > 2
    assert all(torch.equal(x[0]["src"], y[0]["src"]) for x, y in zip(a, b))
    assert any(not torch.equal(x[0]["src"], y[0]["src"]) for x, y in zip(a, c))


def test_native_lookup_varints_padding_and_hardware_crc(tmp_path):
    import ctypes as C
    lib = R.io_lib()
    rng = np.random.default_rng(3)
    # the SSE4.2 path and the portable table path agree (odd alignments and lengths)
    blob = rng.integers(0, 256, 70001, dtype=np.uint8)
    for a, n in ((0, 0), (1, 7), (3, 64), (5, 1001), (0, 70001), (7, 69990)):
        view = blob[a:a + n]
        assert lib.b200st_crc32c(0, view.ctypes.data, n) == lib.b200st_crc32c_table(0, view.ctypes.data, n) == R.crc32c(view.tobytes())
    # records written by TensorFlow: native lookup == general decoder
    for g in GOLD["records"]:
        raw = np.frombuffer(bytes.fromhex(g["framed_hex"]), np.uint8)
        rec = raw[12:-4]
        fast = R.FeatureLookup({"feature": R.VarLenInt64, "label": R.VarLenInt64, "absent": R.VarLenFloat})(rec)
        assert fast["feature"].tolist() == g["ids"]["feature"] and fast["label"].tolist() == g["ids"]["label"] and fast["absent"].size == 0
    # random examples: floats zero-copy, negative / 10-byte varints, single bytes value, empty lists, schema mismatch, fall-backs
    schema = {"audio": R.VarLenFloat, "transcript": R.VarLenInt64, "uuid": R.VarLenString, "src_lang": R.VarLenString, "none": R.VarLenInt64}
    look = R.FeatureLookup(schema)
    for _ in range(20):
        n = int(rng.integers(0, 300))
        ids = rng.integers(-2 ** 62, 2 ** 62, int(rng.integers(0, 40))).astype(np.int64)
        ex = {"audio": rng.standard_normal(n * 80).astype(np.float32), "transcript": ids, "uuid": "u%d" % n, "src_lang": "en",
              "other": np.arange(5)}
        rec = np.frombuffer(R.encode_example(ex), np.uint8)
        fast, slow = look(rec), R.to_dense(R.parse_example(rec), schema)
        assert set(fast) == set(slow)
        assert np.array_equal(fast["audio"], slow["audio"]) and np.array_equal(fast["transcript"], slow["transcript"])
        assert fast["uuid"] == slow["uuid"] == [b"u%d" % n] and fast["none"].size == 0
        assert n == 0 or fast["audio"].base is not None                     # a view of the record, not a copy
    two = np.frombuffer(R.encode_example({"uuid": [b"a", b"b"], "audio": np.ones(2, np.float32)}), np.uint8)
    assert look(two) is None                                                # several bytes values -> general decoder
    unpacked = np.frombuffer(R._ld(1, R._ld(1, R._ld(1, b"transcript") + R._ld(2, R._ld(3, b"\x08\x07\x08\x81\x01")))), np.uint8)
    assert look(unpacked) is None and R.parse_example(unpacked)["transcript"][1].tolist() == [7, 129]
    with pytest.raises(R.TFRecordError):
        R.FeatureLookup({"audio": R.VarLenInt64})(np.frombuffer(R.encode_example({"audio": np.ones(3, np.float32)}), np.uint8))
    with pytest.raises(R.TFRecordError):
        look(np.frombuffer(R.encode_example({"audio": np.ones(3, np.float32)})[:-3], np.uint8))
    # load_tfrecords takes the general decoder for such records and still yields the same elements
    p = tmp_path / "mixed.tfrecords"
    with R.TFRecordWriter(str(p)) as w:
        w.write(R.encode_example({"uuid": [b"a", b"b"], "audio": np.ones(2, np.float32)}))
        w.write(R.encode_example({"uuid": "c", "audio": np.zeros(1, np.float32)}))
    got = list(R.load_tfrecords(str(p), {"audio": R.VarLenFloat, "uuid": R.VarLenString}))
    assert got[0]["uuid"] == [b"a", b"b"] and got[1]["uuid"] == [b"c"] and got[0]["audio"].tolist() == [1.0, 1.0]
    # padded rows
    B, W = 5, 37
    rows = [torch.randn(int(k)) for k in (0, 1, 20, 37, 36)]
    dst = torch.full((B, W), 7.0)
    ptrs = (C.c_void_p * B)(*[r.data_ptr() for r in rows])
    lens = (C.c_int64 * B)(*[r.numel() for r in rows])
    lib.b200st_pad_rows_f32(dst.data_ptr(), W, ptrs, lens, B)
    for j, r in enumerate(rows):
        assert torch.equal(dst[j, :r.numel()], r) and float(dst[j, r.numel():].abs().sum()) == 0.0
