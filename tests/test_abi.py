"""CPU-side checks of the C-ABI boundary: the shared library loads, exports every symbol include/b200st.h
declares, and the host-only entry points (handle, parameter table, workspace planning) behave."""
import ctypes as C
import math
import os
import re

from neurst_b200 import lib as L
from neurst_b200.runtime import make_config
from oracle import restatement as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "b200st.h")).read()
    declared = set(re.findall(r"\b(b200st_[a-z0-9_]+)\s*\(", header))
    lib = L.load()
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert declared == set(L.EXPORTS), declared ^ set(L.EXPORTS)
    assert lib.b200st_version() == L.ABI_VERSION


def test_library_reads_only_measurement_environment_variables():
    """Environment variables may switch on measurement (ablation, PDL off for per-kernel attribution, the GEMM profile
    CSV) or cap NCCL's CTAs, never choose between implementations: every other path would be untested."""
    csrc = os.path.join(ROOT, "neurst_b200", "csrc")
    args = []
    for f in os.listdir(csrc):
        if f.endswith((".cu", ".cuh", ".c")):
            args += re.findall(r"\bgetenv\(\s*([^)]*?)\s*\)", open(os.path.join(csrc, f)).read())
    names = {a[1:-1] for a in args if re.fullmatch(r'"[^"]+"', a)}
    assert len(names) == len(set(args)), "getenv with a non-literal name: %s" % args
    assert names == {"B200ST_ABLATE", "B200ST_NO_PDL", "B200ST_PROFILE_CSV", "B200ST_NCCL_MAX_CTAS"}


def test_io_library_exports_every_declared_symbol():
    import ctypes
    from neurst_b200.csrc import build as B
    header = open(os.path.join(ROOT, "include", "b200st_io.h")).read()
    declared = set(re.findall(r"\b(b200st_[a-z0-9_]+)\s*\(", header))
    assert declared == {"b200st_io_version", "b200st_crc32c", "b200st_crc32c_table", "b200st_crc32c_mask", "b200st_tfrecord_index",
                        "b200st_tfrecord_frame", "b200st_example_lookup", "b200st_decode_varints", "b200st_pad_rows_f32"}
    lib = ctypes.CDLL(B.build_io())
    for sym in declared:
        assert hasattr(lib, sym), sym


def test_parameter_table_matches_reference_layouts():
    lib = L.load()
    for name in ("speech_transformer_toy", "speech_transformer_s", "speech_transformer_m"):
        cfg = R.CONFIGS[name]
        c = make_config(L.MODEL_SPEECH, cfg["d"], cfg["heads"], cfg["ffn"], cfg["enc_layers"], cfg["dec_layers"], cfg["vocab"],
                        channels=cfg["channels"], precision="fp32")
        h = C.c_void_p()
        L.check(lib.b200st_create(C.byref(c), C.byref(h)))
        buf = C.create_string_buffer(128)
        off, nd, shp = C.c_int64(), C.c_int32(), (C.c_int64 * 4)()
        got = []
        for i in range(lib.b200st_param_count(h)):
            L.check(lib.b200st_param_info(h, i, buf, 128, C.byref(off), C.byref(nd), shp))
            assert off.value % 8 == 0
            got.append((buf.value.decode(), tuple(shp[k] for k in range(nd.value))))
        assert got == [(k, tuple(v)) for k, v in R.param_shapes(cfg).items()]
        if name == "speech_transformer_s":
            # 29.26 M parameters, 280 tensors (SURVEY.md §2.2)
            assert len(got) == 280 and sum(math.prod(s) for _, s in got) == 29264384
        lib.b200st_destroy(h)


def test_workspace_planning_and_errors():
    lib = L.load()
    cfg = R.CONFIGS["speech_transformer_s"]
    c = make_config(L.MODEL_SPEECH, cfg["d"], cfg["heads"], cfg["ffn"], cfg["enc_layers"], cfg["dec_layers"], cfg["vocab"],
                    channels=cfg["channels"], precision="bf16", attention_dropout=0.1, ffn_dropout=0.1, postprocess_dropout=0.1)
    h = C.c_void_p()
    L.check(lib.b200st_create(C.byref(c), C.byref(h)))
    train = lib.b200st_workspace_bytes(h, 32, 1000, 88, 1)
    infer = lib.b200st_workspace_bytes(h, 32, 1000, 88, 0)
    assert 0 < infer < train < 16 * 2 ** 30
    lib.b200st_destroy(h)
    bad = make_config(L.MODEL_SPEECH, 250, 4, 64, 1, 1, 10, channels=8, precision="fp32")   # 250 % 4 != 0
    h2 = C.c_void_p()
    assert lib.b200st_create(C.byref(bad), C.byref(h2)) != 0
    assert b"divisible" in lib.b200st_last_error()
    bad2 = make_config(L.MODEL_SPEECH, 36, 4, 64, 1, 1, 10, channels=8, precision="bf16")   # head dim 9 not % 8
    assert lib.b200st_create(C.byref(bad2), C.byref(h2)) != 0


def test_struct_layouts_match_the_c_header(tmp_path):
    """include/b200st.h compiles as plain C (gcc, no CUDA headers) and every struct the ctypes binding mirrors has the
    same size and field offsets as the C definition — the drop-in boundary cannot drift silently."""
    import ctypes as C
    import subprocess
    pairs = [("b200st_operand", L.Operand), ("b200st_gemm_args", L.GemmArgs), ("b200st_config", L.Config),
             ("b200st_buffers", L.Buffers), ("b200st_batch", L.Batch), ("b200st_optim_args", L.OptimArgs),
             ("b200st_step_opts", L.StepOpts), ("b200st_decode_state", L.DecodeState), ("b200st_greedy_args", L.GreedyArgs)]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "b200st.h"', 'int main(void) {']
    for cname, cls in pairs:
        lines.append('  printf("%s.sizeof %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('  printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", inc, str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, cls in pairs:
        assert int(got[cname + ".sizeof"]) == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got["%s.%s" % (cname, fname)]) == getattr(cls, fname).offset, (cname, fname)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """No fallback: without the shared library the binding raises instead of degrading to any CPU / eager path, and a
    Runtime refuses a non-CUDA device."""
    import pytest
    from neurst_b200 import lib as libmod
    monkeypatch.setattr(libmod, "_lib", None)
    monkeypatch.setattr(libmod, "_LIB_PATH", str(tmp_path / "libb200st_missing.so"))
    with pytest.raises(libmod.B200STError):
        libmod.load(build_if_missing=False)
    monkeypatch.undo()
    from neurst_b200.runtime import Runtime
    cfg = make_config(L.MODEL_SPEECH, 16, 2, 32, 1, 1, 32, channels=8, feat=80, in_channels=1)
    with pytest.raises(L.B200STError):
        Runtime(cfg, device="cpu")
