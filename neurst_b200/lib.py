"""ctypes binding of libb200st.so (the C-ABI boundary declared in include/b200st.h).

The product path has NO fallback: if the shared library is missing or a call fails, an exception is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libb200st.so")
_lib = None

F32, BF16, F16 = 0, 1, 2
ABI_VERSION = 201    # must equal b200st_version(): bumped whenever a struct in include/b200st.h changes layout


class B200STError(RuntimeError):
    pass


class Operand(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("dtype", C.c_int32), ("mn_major", C.c_int32),
                ("ld", C.c_int64), ("sb1", C.c_int64), ("sb2", C.c_int64)]


class GemmArgs(C.Structure):
    _fields_ = [("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("nb1", C.c_int32), ("nb2", C.c_int32),
                ("A", Operand), ("B", Operand),
                ("C", C.c_void_p), ("c_dtype", C.c_int32), ("ldc", C.c_int64), ("c_sb1", C.c_int64),
                ("c_sb2", C.c_int64),
                ("alpha", C.c_float), ("bias", C.c_void_p), ("relu", C.c_int32),
                ("mask_src", C.c_void_p), ("mask_dtype", C.c_int32), ("mask_ld", C.c_int64),
                ("mask_sb1", C.c_int64), ("mask_sb2", C.c_int64),
                ("dropout_p", C.c_float), ("dropout_seed", C.c_uint64), ("dropout_stream", C.c_uint64),
                ("residual", C.c_void_p), ("res_ld", C.c_int64), ("res_sb1", C.c_int64), ("res_sb2", C.c_int64),
                ("accumulate", C.c_int32), ("splitk", C.c_int32), ("force_simt", C.c_int32)]


def lib_path():
    return _LIB_PATH


def load(build_if_missing=True):
    """Loads libb200st.so, building it with nvcc when the in-tree binary is absent/stale and nvcc exists."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        from neurst_b200.csrc import build as _build
        try:
            _build.build()          # no-op when the in-tree binary matches the source digest; locked + atomic otherwise
        except Exception as e:  # noqa
            # a stale or missing library never loads silently: its struct layouts may no longer match the ctypes mirror
            raise B200STError("libb200st.so is missing or stale and could not be (re)built: %s" % e)
    if not os.path.exists(_LIB_PATH):
        raise B200STError("libb200st.so not found at %s (run `python -m neurst_b200.csrc.build`)" % _LIB_PATH)
    lib = C.CDLL(_LIB_PATH)
    lib.b200st_last_error.restype = C.c_char_p
    lib.b200st_version.restype = C.c_int
    if lib.b200st_version() != ABI_VERSION:
        raise B200STError("libb200st.so ABI version %d != binding version %d" % (lib.b200st_version(), ABI_VERSION))
    lib.b200st_launch_count.restype = C.c_int64
    _declare(lib)
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise B200STError(load().b200st_last_error().decode("utf-8", "replace"))


def launch_count():
    return int(load().b200st_launch_count())


def _dt(t):
    import torch
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    if t.dtype == torch.float16:
        return F16
    raise B200STError("unsupported dtype %s" % t.dtype)


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _gemm_args(A, B, Cout, a_mn=False, b_mn=False, alpha=1.0, bias=None, relu=False, mask_src=None, dropout=None,
               residual=None, accumulate=False, splitk=1, force_simt=False):

    def norm(t):
        while t.dim() < 4:
            t = t.unsqueeze(0)
        assert t.stride(-1) == 1
        return t

    A4, B4, C4 = norm(A), norm(B), norm(Cout)
    g = GemmArgs()
    M, N = C4.shape[-2], C4.shape[-1]
    K = A4.shape[-2] if a_mn else A4.shape[-1]
    g.M, g.N, g.K = M, N, K
    g.nb2, g.nb1 = C4.shape[0], C4.shape[1]
    g.A = Operand(A4.data_ptr(), _dt(A4), int(a_mn), A4.stride(-2), A4.stride(1), A4.stride(0))
    g.B = Operand(B4.data_ptr(), _dt(B4), int(b_mn), B4.stride(-2), B4.stride(1), B4.stride(0))
    g.C, g.c_dtype, g.ldc, g.c_sb1, g.c_sb2 = C4.data_ptr(), _dt(C4), C4.stride(-2), C4.stride(1), C4.stride(0)
    g.alpha = alpha
    g.bias = bias.data_ptr() if bias is not None else None
    g.relu = int(relu)
    if mask_src is not None:
        m4 = norm(mask_src)
        g.mask_src, g.mask_dtype = m4.data_ptr(), _dt(m4)
        g.mask_ld, g.mask_sb1, g.mask_sb2 = m4.stride(-2), m4.stride(1), m4.stride(0)
    if dropout is not None:
        g.dropout_p, g.dropout_seed, g.dropout_stream = dropout
    if residual is not None:
        r4 = norm(residual)
        g.residual = r4.data_ptr()
        g.res_ld, g.res_sb1, g.res_sb2 = r4.stride(-2), r4.stride(1), r4.stride(0)
    g.accumulate = int(accumulate)
    g.splitk = splitk
    g.force_simt = int(force_simt)
    return g


def gemm(A, B, Cout, **kw):
    """Generic contraction on 2-D/3-D/4-D torch CUDA tensors (tests & glue).

    A: [..., M, K] (K-major) or [..., K, M] (a_mn); B: [..., N, K] or [..., K, N] (b_mn); Cout: [..., M, N].
    Leading dims (0, 1 or 2 of them) are batch dims; inner dim must be contiguous.
    """
    g = _gemm_args(A, B, Cout, **kw)
    check(load().b200st_gemm(C.byref(g), _stream()))
    return Cout


def gemm_bench(A, B, Cout, iters=50, **kw):
    """ms per launch of one GEMM, timed with CUDA events inside the library (no Python overhead)."""
    g = _gemm_args(A, B, Cout, **kw)
    ms = C.c_float(0)
    check(load().b200st_gemm_bench(C.byref(g), iters, C.byref(ms), _stream()))
    return ms.value


# ------------------------------------------------------------------------------------------------
# model-level structs (mirror include/b200st.h)
# ------------------------------------------------------------------------------------------------
MODEL_SPEECH, MODEL_TEXT, MODEL_ENCODER, MODEL_DECODER, MODEL_MHA = 0, 1, 2, 3, 4


class Config(C.Structure):
    _fields_ = [("model_type", C.c_int32),
                ("d", C.c_int32), ("heads", C.c_int32), ("ffn", C.c_int32), ("enc_layers", C.c_int32),
                ("dec_layers", C.c_int32), ("vocab", C.c_int32), ("src_vocab", C.c_int32),
                ("feat", C.c_int32), ("in_channels", C.c_int32), ("channels", C.c_int32), ("conv_layer_norm", C.c_int32),
                ("precision", C.c_int32),
                ("ln_eps", C.c_float), ("attention_dropout", C.c_float), ("ffn_dropout", C.c_float),
                ("postprocess_dropout", C.c_float), ("label_smoothing", C.c_float),
                ("share_src_trg_embedding", C.c_int32),
                ("mha_self", C.c_int32), ("mha_din", C.c_int32), ("mha_dmem", C.c_int32), ("mha_dout", C.c_int32),
                ("with_cross_attention", C.c_int32), ("disable_fused_attention", C.c_int32), ("deterministic", C.c_int32)]


class Buffers(C.Structure):
    _fields_ = [("params", C.c_void_p), ("shadow", C.c_void_p), ("grads", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_uint64)]


class Batch(C.Structure):
    _fields_ = [("src", C.c_void_p), ("src_ids", C.c_void_p), ("src_length", C.c_void_p), ("src_padding", C.c_void_p),
                ("trg_input", C.c_void_p), ("trg", C.c_void_p), ("trg_length", C.c_void_p),
                ("B", C.c_int32), ("T", C.c_int32), ("L", C.c_int32), ("training", C.c_int32),
                ("seed", C.c_uint64), ("seed_dev", C.c_void_p), ("loss_scale", C.c_float), ("loss_scale_dev", C.c_void_p),
                ("logits", C.c_void_p), ("loss", C.c_void_p), ("nll_sum", C.c_void_p), ("n_tokens", C.c_void_p),
                ("enc_out", C.c_void_p)]


class OptimArgs(C.Structure):
    _fields_ = [("params", C.c_void_p), ("grads", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p),
                ("shadow", C.c_void_p), ("shadow_dtype", C.c_int32), ("numel", C.c_int64),
                ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("step_t", C.c_int64), ("grad_scale", C.c_float), ("zero_grad", C.c_int32),
                ("clip_value", C.c_float), ("clip_norm", C.c_float),
                ("tensor_sumsq", C.c_void_p), ("loss_scale_state", C.c_void_p),
                ("growth_steps", C.c_float), ("multiplier", C.c_float)]


class StepOpts(C.Structure):
    _fields_ = [("allreduce_grads", C.c_int32), ("optim", C.POINTER(OptimArgs))]


class DecodeState(C.Structure):
    _fields_ = [("B", C.c_int32), ("Tm", C.c_int32), ("max_len", C.c_int32),
                ("cross_kv", C.c_void_p), ("self_kv", C.c_void_p), ("memory_bias", C.c_void_p), ("scratch", C.c_void_p),
                ("use_shadow", C.c_int32)]


class GreedyArgs(C.Structure):
    _fields_ = [("bos_ids", C.c_void_p), ("eos_id", C.c_int32), ("unk_id", C.c_int32), ("min_len", C.c_int32),
                ("max_steps", C.c_int32), ("out_ids", C.c_void_p), ("out_len", C.c_void_p), ("out_logprob", C.c_void_p),
                ("state_words", C.c_void_p), ("use_graph", C.c_int32)]


# every symbol include/b200st.h declares (tests/test_abi.py checks the .so exports all of them)
EXPORTS = [
    "b200st_last_error", "b200st_version", "b200st_launch_count", "b200st_gemm", "b200st_gemm_bench", "b200st_profile_begin", "b200st_profile_end",
    "b200st_create", "b200st_destroy", "b200st_param_arena_numel", "b200st_param_count", "b200st_param_info",
    "b200st_workspace_bytes", "b200st_forward", "b200st_forward_backward", "b200st_refresh_shadow", "b200st_adam_step", "b200st_optimizer_step",
    "b200st_comm_unique_id", "b200st_comm_init", "b200st_comm_broadcast", "b200st_comm_destroy", "b200st_comm_stats", "b200st_train_step",
    "b200st_encode", "b200st_encode_workspace_bytes", "b200st_decode_scratch_floats", "b200st_decode_init", "b200st_decode_step",
    "b200st_greedy_search", "b200st_greedy_used_graph",
    "b200st_encoder_forward", "b200st_decoder_forward", "b200st_mha_forward", "b200st_lsce", "b200st_layernorm_fwd",
    "b200st_layernorm_bwd", "b200st_softmax_fwd", "b200st_conv1_ln_relu_fwd", "b200st_dropout_stream_id", "b200st_dropout_mask",
    "b200st_attention_fwd", "b200st_attention_bwd", "b200st_ffn_fwd", "b200st_ffn_bwd",
]


def _declare(lib):
    lib.b200st_param_arena_numel.restype = C.c_int64
    lib.b200st_param_arena_numel.argtypes = [C.c_void_p]
    lib.b200st_param_count.restype = C.c_int32
    lib.b200st_param_count.argtypes = [C.c_void_p]
    lib.b200st_workspace_bytes.restype = C.c_int64
    lib.b200st_workspace_bytes.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    lib.b200st_dropout_stream_id.restype = C.c_uint64
    lib.b200st_dropout_stream_id.argtypes = [C.c_char_p]
    lib.b200st_destroy.argtypes = [C.c_void_p]
    lib.b200st_param_info.argtypes = [C.c_void_p, C.c_int32, C.c_char_p, C.c_int32, C.POINTER(C.c_int64),
                                      C.POINTER(C.c_int32), C.POINTER(C.c_int64)]
    lib.b200st_forward.argtypes = [C.c_void_p, C.POINTER(Buffers), C.POINTER(Batch), C.c_void_p]
    lib.b200st_forward_backward.argtypes = [C.c_void_p, C.POINTER(Buffers), C.POINTER(Batch), C.c_void_p]
    lib.b200st_refresh_shadow.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p]
    lib.b200st_optimizer_step.argtypes = [C.c_void_p, C.POINTER(OptimArgs), C.c_void_p]
    lib.b200st_comm_unique_id.argtypes = [C.c_char_p]
    lib.b200st_comm_init.argtypes = [C.c_void_p, C.c_char_p, C.c_int32, C.c_int32]
    lib.b200st_comm_broadcast.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
    lib.b200st_comm_destroy.argtypes = [C.c_void_p]
    lib.b200st_comm_stats.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.b200st_train_step.argtypes = [C.c_void_p, C.POINTER(Buffers), C.POINTER(Batch), C.POINTER(StepOpts), C.c_void_p]
    lib.b200st_encode.argtypes = [C.c_void_p, C.POINTER(Buffers), C.POINTER(Batch), C.c_void_p, C.c_void_p, C.c_void_p]
    lib.b200st_encode_workspace_bytes.restype = C.c_int64
    lib.b200st_encode_workspace_bytes.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    lib.b200st_decode_scratch_floats.restype = C.c_int64
    lib.b200st_decode_scratch_floats.argtypes = [C.c_void_p, C.c_int32]
    lib.b200st_decode_init.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_void_p, C.POINTER(DecodeState), C.c_void_p]
    lib.b200st_decode_step.argtypes = [C.c_void_p, C.POINTER(Buffers), C.POINTER(DecodeState), C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]
    lib.b200st_greedy_search.argtypes = [C.c_void_p, C.POINTER(Buffers), C.POINTER(DecodeState), C.POINTER(GreedyArgs),
                                         C.c_void_p]
    lib.b200st_adam_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float,
                                     C.c_float, C.c_float, C.c_float, C.c_int64, C.c_float, C.c_int32, C.c_void_p]
    lib.b200st_encoder_forward.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                           C.c_void_p, C.c_int32, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)]
    lib.b200st_decoder_forward.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                           C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_uint64, C.c_void_p,
                                           C.POINTER(C.c_uint64)]
    lib.b200st_mha_forward.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                       C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
    lib.b200st_lsce.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_void_p]
    lib.b200st_layernorm_fwd.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_int32,
                                         C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]
    lib.b200st_layernorm_bwd.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                                         C.c_int32, C.c_int32, C.c_void_p]
    lib.b200st_softmax_fwd.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int64,
                                       C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    lib.b200st_dropout_mask.argtypes = [C.c_uint64, C.c_uint64, C.c_int64, C.c_float, C.c_void_p, C.c_void_p]
    lib.b200st_attention_fwd.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                         C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                         C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    lib.b200st_attention_bwd.argtypes = [C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                         C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                         C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                         C.c_void_p]
    lib.b200st_ffn_fwd.argtypes = [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_float, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]
    lib.b200st_ffn_bwd.argtypes = [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]
    lib.b200st_gemm.argtypes = [C.POINTER(GemmArgs), C.c_void_p]
    lib.b200st_gemm_bench.argtypes = [C.POINTER(GemmArgs), C.c_int32, C.POINTER(C.c_float), C.c_void_p]


def softmax(S, P, bias=None, causal=False):
    """P = softmax(S + bias[b,k] (+ causal mask)) over the last axis; S fp32 [B,H,Tq,Tk] (last dim contiguous)."""
    B, H, Tq, Tk = S.shape
    assert S.stride(-1) == 1 and P.stride(-1) == 1 and S.stride(2) % 8 == 0 and P.stride(2) % 8 == 0, \
        "softmax rows must be padded to a multiple of 8 (use padded_scores())"
    check(load().b200st_softmax_fwd(S.data_ptr(), S.stride(2), bias.data_ptr() if bias is not None else None, int(causal),
                                    P.data_ptr(), _dt(P), P.stride(2), B, H, Tq, Tk, _stream()))
    return P


def layernorm(x, gamma, beta, eps, out_dtype=None, relu=False):
    """LayerNorm over the last axis of a contiguous tensor (fp32 or bf16 in, fp32/bf16 out)."""
    import torch
    cols = x.shape[-1]
    rows = x.numel() // cols
    y = torch.empty(x.shape, dtype=out_dtype or x.dtype, device=x.device)
    check(load().b200st_layernorm_fwd(x.data_ptr(), _dt(x), gamma.data_ptr(), beta.data_ptr(), eps, y.data_ptr(), _dt(y),
                                      None, None, rows, cols, int(relu), _stream()))
    return y


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _rows(t, cols=None):
    """(rows, row stride) of a 2-D row view with a unit inner stride (a column slice of a packed buffer is fine)."""
    assert t.dim() == 2 and t.stride(1) == 1, "expected a 2-D view with a contiguous inner dimension"
    assert cols is None or t.shape[1] == cols, (tuple(t.shape), cols)
    return t.shape[0], t.stride(0)


def attention_fwd(q, k, v, ctx, lse, B, H, bias=None, kv_len=None, causal=False, drop_p=0.0, keep_bits=None):
    """Fused attention forward (head dim 64, bf16/fp16).  q, ctx: [B*Tq, H*64] views; k, v: [B*Tk, H*64] views; lse fp32
    [B, H, Tq]; bias fp32 [B, Tk]; kv_len int32 [B]; keep_bits uint8 [B*H*Tq*round8(Tk) / 8] (bit j of byte g = element
    8g+j).  Writes ctx and lse."""
    nq, q_ld = _rows(q, H * 64)
    nk, k_ld = _rows(k, H * 64)
    _, v_ld = _rows(v, H * 64)
    _, ctx_ld = _rows(ctx, H * 64)
    check(load().b200st_attention_fwd(_dt(q), q.data_ptr(), q_ld, k.data_ptr(), k_ld, v.data_ptr(), v_ld, B, H, nq // B, nk // B,
                                      _ptr(bias), _ptr(kv_len), int(causal), drop_p, _ptr(keep_bits), ctx.data_ptr(), ctx_ld,
                                      lse.data_ptr(), _stream()))
    return ctx, lse


def attention_bwd(q, k, v, ctx, dctx, lse, dq, dk, dv, dq_scratch, B, H, bias=None, kv_len=None, causal=False, drop_p=0.0,
                  keep_bits=None):
    """Fused attention backward: dq [B*Tq, H*64], dk / dv [B*Tk, H*64] views written from ctx / lse of the forward pass
    and dctx; dq_scratch fp32 with B*Tq*H*64 + B*H*Tq elements."""
    nq, q_ld = _rows(q, H * 64)
    nk, k_ld = _rows(k, H * 64)
    _, v_ld = _rows(v, H * 64)
    _, ctx_ld = _rows(ctx, H * 64)
    _, dctx_ld = _rows(dctx, H * 64)
    _, dq_ld = _rows(dq, H * 64)
    _, dk_ld = _rows(dk, H * 64)
    _, dv_ld = _rows(dv, H * 64)
    Tq = nq // B
    assert dq_scratch.dtype.itemsize == 4 and dq_scratch.numel() >= B * Tq * H * 64 + B * H * Tq
    check(load().b200st_attention_bwd(_dt(q), q.data_ptr(), q_ld, k.data_ptr(), k_ld, v.data_ptr(), v_ld, B, H, Tq, nk // B,
                                      _ptr(bias), _ptr(kv_len), int(causal), drop_p, _ptr(keep_bits), ctx.data_ptr(), ctx_ld,
                                      dctx.data_ptr(), dctx_ld, lse.data_ptr(), dq_scratch.data_ptr(), dq.data_ptr(), dq_ld,
                                      dk.data_ptr(), dk_ld, dv.data_ptr(), dv_ld, _stream()))
    return dq, dk, dv


def ffn_fwd(X, W1, b1, W2, b2, F1, x_out, drop_ffn_p=0.0, ffn_bits=None, drop_post_p=0.0, post_bits=None, tickets=None):
    """Fused FFN forward on packed row-major tensors: F1 [M, ffn] = dropout(relu(X W1 + b1)); x_out fp32 [M, d] +=
    post-dropout(F1 W2 + b2).  X [M, d], W1 [d, ffn], W2 [ffn, d] bf16/fp16.  Returns the number of hidden slices."""
    M, d = X.shape
    ffn = W1.shape[1]
    for t in (X, W1, W2, F1, x_out):
        assert t.is_contiguous()
    splits = C.c_int32(0)
    check(load().b200st_ffn_fwd(_dt(X), X.data_ptr(), M, d, ffn, W1.data_ptr(), _ptr(b1), W2.data_ptr(), _ptr(b2), drop_ffn_p,
                                _ptr(ffn_bits), drop_post_p, _ptr(post_bits), F1.data_ptr(), x_out.data_ptr(), _ptr(tickets),
                                C.byref(splits), _stream()))
    return splits.value


def ffn_bwd(dY, W1, W2, F1, scale, dF1, dH, tickets=None):
    """Fused FFN data gradient: dF1 [M, ffn] = scale * (dY W2^T) where F1 > 0; dH fp32 [M, d] += dF1 W1^T.
    Returns the number of hidden slices."""
    M, d = dY.shape
    ffn = W1.shape[1]
    for t in (dY, W1, W2, F1, dF1, dH):
        assert t.is_contiguous()
    splits = C.c_int32(0)
    check(load().b200st_ffn_bwd(_dt(dY), dY.data_ptr(), M, d, ffn, W1.data_ptr(), W2.data_ptr(), F1.data_ptr(), scale,
                                dF1.data_ptr(), dH.data_ptr(), _ptr(tickets), C.byref(splits), _stream()))
    return splits.value


def profile_begin():
    check(load().b200st_profile_begin())


def profile_end():
    """-> (sum of tcgen05 GEMM kernel ms, sum of their algorithmic FLOPs, launches) since profile_begin()."""
    ms, fl, n = C.c_double(0), C.c_double(0), C.c_int64(0)
    check(load().b200st_profile_end(C.byref(ms), C.byref(fl), C.byref(n)))
    return ms.value, fl.value, n.value


def padded_scores(B, H, Tq, Tk, dtype, device):
    """[B,H,Tq,Tk] view of a buffer whose rows are padded to a multiple of 8 (softmax / TMA row-stride rule)."""
    import torch
    Tkp = (Tk + 7) // 8 * 8
    return torch.zeros(B, H, Tq, Tkp, dtype=dtype, device=device)[..., :Tk]
