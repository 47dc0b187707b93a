"""ctypes door to oracle/_ref/libdashinfer_ref.so — the UNMODIFIED reference GPU code (span-attention library + the
span-cache writers) built by oracle/build_ref.py.  TEST INFRASTRUCTURE: only tests/golden/make_ref_pin.py imports this.

    load() -> lib or None          (None when the library was never built)
    span_attn(lib, out, q, k_tab, v_tab, lens_host, nH, nG, span, n_spans, qmode, scale)
    cache_append(lib, k_tab, v_tab, q_out, qkv, old_lens_u32, nH, nG, span, n_spans, qmode)
    context_span_copy(lib, span_ptrs, src, nG, span, seq_len, qmode)
All tensors are torch CUDA tensors; dtype bf16 (span::DataType::BF16 = 2) or fp16 (1).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_ref", "libdashinfer_ref.so")
_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO):
        return None
    lib = C.CDLL(SO)
    vp, i32, f32 = C.c_void_p, C.c_int, C.c_float
    lib.ref_span_attn.restype = i32
    lib.ref_span_attn.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, f32, vp]
    lib.ref_cache_append.restype = i32
    lib.ref_cache_append.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp]
    lib.ref_context_span_copy.restype = i32
    lib.ref_context_span_copy.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp]
    lib.ref_version.restype = C.c_char_p
    _lib = lib
    return lib


def _dt(t):
    import torch
    return {torch.float16: 1, torch.bfloat16: 2}[t.dtype]


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def span_attn(lib, out, q, k_tab, v_tab, lens_host, n_heads, n_groups, span, n_spans, qmode, scale, head=128):
    import numpy as np
    lens = np.ascontiguousarray(np.asarray(lens_host, dtype=np.int32))
    rc = lib.ref_span_attn(out.data_ptr(), q.data_ptr(), k_tab.data_ptr(), v_tab.data_ptr(), lens.ctypes.data, len(lens),
                           n_heads, n_groups, head, span, n_spans, qmode, _dt(q), float(scale), _stream())
    assert rc == 0, "reference span::Run failed: %d" % rc
    return out


def cache_append(lib, k_tab, v_tab, q_out, qkv, old_lens, n_heads, n_groups, span, n_spans, qmode, head=128):
    """old_lens: int32/uint32 device tensor [batch] (the reference reads uint32)."""
    rc = lib.ref_cache_append(k_tab.data_ptr(), v_tab.data_ptr(), q_out.data_ptr(), qkv.data_ptr(), old_lens.data_ptr(),
                              qkv.shape[0], n_heads, n_groups, head, span, n_spans, qmode, _dt(qkv), _stream())
    assert rc == 0, "reference DecoderCacheAppendLauncher failed: %d" % rc
    return q_out


def context_span_copy(lib, span_ptrs, src, n_groups, span, seq_len, qmode, head=128):
    """span_ptrs: int64 device tensor of span pointers of ONE sequence; src [seq_len, n_groups, head] contiguous."""
    rc = lib.ref_context_span_copy(span_ptrs.data_ptr(), src.data_ptr(), n_groups, head, span, seq_len, qmode, _dt(src), _stream())
    assert rc == 0, "reference ContextSpanCopyLauncher failed: %d" % rc
