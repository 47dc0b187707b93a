"""Pins the KV-cache half of the oracle — and the b200spark kernels — to the REFERENCE'S OWN GPU code.

The reference's results are stored in tests/golden/ref_pin.json (SHA-256 of every span byte its span-cache writers
produced, and of the Q rows its append gathered) and tests/golden/ref_pin_attn.npz (its span-attention outputs).
tests/golden/make_ref_pin.py made them from the unmodified span-attention library and span-cache writers of
modelscope/dash-infer @ f3cca8e, compiled for sm_100 by oracle/build_ref.py, on the seeded inputs drawn here
(VERDICT r1: "the KV / attention oracle is unpinned ... it could have been compiled for the GPU box as oracle/_ref").

What is pinned, and how tightly:
  * bf16 (QuantMode::NONE) append: byte-identical spans.
  * I8 / U4 append: b200spark repeats the arithmetic the reference kernel executes as compiled (--use_fast_math:
    multiply by fl(1/RANGE), MUFU.RCP, contracted FFMAs, one rint conversion) -> EVERY span byte and every {zero, scale}
    is bit-identical to DecoderCacheAppendLauncher's.  The CPU oracle (oracle/kvcache_ref.py) restates the same formula
    with an IEEE reciprocal in place of MUFU.RCP: identical scales; zero points differ (by 1) only on exact-tie rows
    (max == -min, about 1 % of N(0,1) bf16 rows, half of which fall the other way); measured rates are printed.
  * attention (NONE / I8 / U4) on IDENTICAL cache bytes (b200spark's append must reproduce the digest of the cache the
    reference's append wrote): b200spark vs span::Run vs the fp64 oracle.  The reference stores scores / probabilities
    in bf16 (span_attention.hpp: QK workspace is FType), so it carries ~2^-9 relative error per probability; asserted:
    b200spark is within the oracle tolerance, the reference is within 3e-2 of the oracle, and b200spark is at least as
    close to the oracle as the reference is.
"""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from oracle import kvcache_ref as KV

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_GOLDEN = {}


def _golden():
    if not _GOLDEN:
        with open(os.path.join(GOLDEN, "ref_pin.json")) as f:
            _GOLDEN.update(json.load(f))
        with np.load(os.path.join(GOLDEN, "ref_pin_attn.npz")) as z:
            _GOLDEN["attn_out"] = {k: z[k] for k in z.files}
    return _GOLDEN


def _rows(rng, B, width):
    return torch.from_numpy(rng.standard_normal((B, width)).astype(np.float32)).to(torch.bfloat16).cuda()


def b2_append(cache, qkv, pos):
    from b200spark import ops
    return ops.cache_append(cache, qkv, pos)


def digest(cache, *extra):
    """SHA-256 of every span of every sequence in table order (K spans, then V spans), then of the bytes of `extra`
    tensors: independent of where the pages lie in the pool.  Asserts that no pool byte outside the spans was written
    (every pool here starts filled with 0)."""
    h = hashlib.sha256()
    for pool, perm in ((cache.k_pool, cache.perm_k), (cache.v_pool, cache.perm_v)):
        p = pool.cpu().numpy()
        outside = np.ones(p.size, dtype=bool)
        for off in (perm.flatten() * cache.stride).tolist():
            h.update(p[off:off + cache.span_bytes].tobytes())
            outside[off:off + cache.span_bytes] = False
        assert not p[outside].any(), "bytes written outside the spans"
    for t in extra:
        h.update(t.contiguous().view(torch.uint8).cpu().numpy().tobytes())
    return h.hexdigest()


def append_fill(append, mode, span, B=4, nH=8, nG=2, T=300, max_len=384):
    """Append T tokens of N(0,1) rows to B sequences with `append(cache, qkv, pos) -> q` -> (cache, Q of the last step,
    rows [T, B, width] bf16)."""
    from b200spark import ops
    rng = np.random.default_rng(mode * 10 + span)
    cache = ops.SpanCache(B, max_len, nH, nG, span, mode)
    width = (nH + 2 * nG) * 128
    pos = torch.zeros(B, dtype=torch.int32, device="cuda")
    rows_all = []
    for t in range(T):
        qkv = _rows(rng, B, width)
        rows_all.append(qkv.cpu())
        q = append(cache, qkv, pos)
        pos += 1
    torch.cuda.synchronize()
    return cache, q, torch.stack(rows_all)


def _ulp_diff(a, b):
    ai = a.view(np.int32).astype(np.int64)
    bi = b.view(np.int32).astype(np.int64)
    return np.abs(ai - bi)


def _codes(buf, mode, nG, span, n):
    row = {KV.QUANT_I8: 128, KV.QUANT_U4: 64}[mode]
    d = buf[:nG * span * row].reshape(nG, span, row)[:, :n]
    if mode == KV.QUANT_I8:
        return d.view(np.int8).astype(np.int32)
    return np.stack([d & 0xF, d >> 4], -1).reshape(nG, n, 128).astype(np.int32)


MODES = [KV.QUANT_NONE, KV.QUANT_I8, KV.QUANT_U4]
APPEND_SPANS = [16, 32, 64, 128]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("span", APPEND_SPANS)
def test_append_bit_exact_against_reference_kernel(mode, span):
    """300 tokens x 4 sequences x (8 + 2 x 2) heads through b2_span_cache_append: EVERY byte of every span (codes and
    {zero, scale} params) and the gathered Q must be identical to what DecoderCacheAppendLauncher wrote into identically
    laid out page tables.  The CPU oracle is compared with the same bytes and its (tie-row) deviation is recorded."""
    B, nH, nG, T = 4, 8, 2, 300
    cb, q, rows = append_fill(b2_append, mode, span, B, nH, nG, T)
    assert digest(cb, q) == _golden()["append"]["mode%d_span%d" % (mode, span)], "span bytes differ from the reference kernel's"
    # ---- the oracle against the same (reference) bytes
    oref = {w: KV.SpanCacheRef(mode, span, nG) for w in "kv"}
    for w in "kv":
        for _ in range(B):
            oref[w].add_sequence()
    x = rows.float().numpy().reshape(T, B, nH + 2 * nG, 128)
    for t in range(T):
        for b in range(B):
            oref["k"].append(b, t, x[t, b, nH:nH + nG]); oref["v"].append(b, t, x[t, b, nH + nG:])
    n_rows = z_bad = n_codes = c_bad = c_bad_same_zero = 0
    for b in range(B):
        for si in range((T + span - 1) // span):
            n = min(span, T - si * span)
            for which in "kv":
                r = cb.span_view(which, b, si).cpu().numpy()
                o = oref[which].spans[b][si]
                if mode == KV.QUANT_NONE:
                    assert np.array_equal(r.reshape(nG, span, 256)[:, :n], o.reshape(nG, span, 256)[:, :n])
                    continue
                row = {KV.QUANT_I8: 128, KV.QUANT_U4: 64}[mode]
                rp = r[nG * span * row:].view(np.float32).reshape(nG, span, 2)[:, :n]
                op = o[nG * span * row:].view(np.float32).reshape(nG, span, 2)[:, :n]
                assert np.array_equal(rp[..., 1], op[..., 1]), "oracle scale must equal the reference's bit for bit"
                dz = np.abs(rp[..., 0] - op[..., 0])
                assert dz.max() <= 1.0
                dc = np.abs(_codes(r, mode, nG, span, n) - _codes(o, mode, nG, span, n))
                same = dz == 0
                assert dc.max() <= 2 and dc[same].max(initial=0) <= 1
                n_rows += dz.size; z_bad += int((~same).sum()); n_codes += dc.size
                c_bad += int((dc != 0).sum()); c_bad_same_zero += int((dc[same] != 0).sum())
    if mode == KV.QUANT_NONE:
        return
    print("oracle vs reference append, mode %d span %d: zero differs on %d / %d rows, codes differ %d / %d (%d where the zero agrees)"
          % (mode, span, z_bad, n_rows, c_bad, n_codes, c_bad_same_zero))
    assert z_bad / n_rows < 3e-2 and c_bad_same_zero / n_codes < 5e-3


def _oracle_from_device(cache, mode, span, nG, B, lens):
    """SpanCacheRef holding the exact bytes of a device cache (so all three implementations read the same cache)."""
    ref = {w: KV.SpanCacheRef(mode, span, nG) for w in "kv"}
    for w in "kv":
        for b in range(B):
            ref[w].add_sequence()
            for si in range((lens[b] + span - 1) // span):
                ref[w].spans[b].append(cache.span_view(w, b, si).cpu().numpy().copy())
    return ref["k"], ref["v"]


CASES = [  # (lens, nH, nG, span) — the reference's own shapes (test_quant_none.cpp:727-763) + Qwen2-7B geometry
    ([15], 1, 1, 16), ([33], 2, 1, 32), ([15, 16], 2, 1, 32), ([17, 31], 2, 1, 32), ([17], 7, 1, 16), ([3], 4, 2, 16),
    ([17, 15], 16, 2, 16), ([81, 99, 133, 255], 16, 2, 16), ([1, 63, 64, 65, 200, 777], 28, 4, 128), ([2049, 300], 28, 4, 64),
]
ATTN_SCALE = 1.0 / np.sqrt(128)


def attention_fill(append, mode, case):
    """The cache of CASES[case]: max(lens) steps of N(0,1) rows, finished sequences writing past their end ->
    (cache, the Q of every sequence's last token)."""
    from b200spark import ops
    lens, nH, nG, span = CASES[case]
    B, T = len(lens), max(lens)
    max_len = (T + span) // span * span
    rng = np.random.default_rng(case * 3 + mode)
    cache = ops.SpanCache(B, max_len, nH, nG, span, mode)
    width = (nH + 2 * nG) * 128
    q_last = torch.zeros(B, nH * 128, dtype=torch.bfloat16, device="cuda")
    for t in range(T):
        qkv = _rows(rng, B, width)
        pos = torch.tensor([min(t, lens[b]) for b in range(B)], dtype=torch.int32, device="cuda")
        q = append(cache, qkv, pos)
        for b in range(B):
            if t == lens[b] - 1:
                q_last[b] = q[b]
    torch.cuda.synchronize()
    return cache, q_last


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", range(len(CASES)))
def test_attention_against_reference_library(mode, case):
    from b200spark import ops
    lens, nH, nG, span = CASES[case]
    B = len(lens)
    key = "mode%d_case%d" % (mode, case)
    cache, q_last = attention_fill(b2_append, mode, case)
    assert digest(cache, q_last) == _golden()["attention"][key], "cache bytes differ from the ones the reference read"
    attn = ops.SpanAttn(cache.cfg, B)
    out_b2 = attn(q_last, cache, torch.tensor(lens, dtype=torch.int32, device="cuda"), cache.max_len, ops.Workspace(),
                  scale=ATTN_SCALE)
    torch.cuda.synchronize()
    kref, vref = _oracle_from_device(cache, mode, span, nG, B, lens)
    orc = KV.attention_ref(q_last.float().cpu().numpy().reshape(B, nH, 128), kref, vref, lens, nH, ATTN_SCALE)
    b2 = out_b2.float().cpu().numpy().reshape(B, nH, 128)
    rf = KV.bits_to_f32(_golden()["attn_out"][key]).reshape(B, nH, 128)  # span::Run's bf16 output
    e_b2, e_rf, e_x = float(np.abs(b2 - orc).max()), float(np.abs(rf - orc).max()), float(np.abs(b2 - rf).max())
    print("attention mode %d %s: |b2-oracle| %.2e  |ref-oracle| %.2e  |b2-ref| %.2e" % (mode, CASES[case], e_b2, e_rf, e_x))
    assert np.all(np.abs(b2 - orc) <= 2e-3 + 2.0 ** -7 * np.abs(orc)), e_b2
    assert e_rf <= 3e-2, e_rf
    assert e_x <= 3e-2, e_x
    assert e_b2 <= e_rf + 4e-3  # never worse than the reference by more than the bf16 output rounding


CONTEXT_SHAPES = [(16, 64), (32, 96), (64, 64), (128, 384)]


def context_src(mode, span, seq, nG=2):
    rng = np.random.default_rng(seq + span + mode)
    return torch.from_numpy(rng.standard_normal((seq, nG * 128)).astype(np.float32)).to(torch.bfloat16).cuda()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("span,seq", CONTEXT_SHAPES)
def test_context_span_copy_bit_exact_against_reference(mode, span, seq):
    """Prefill-side cache writer (SURVEY.md §8 f4): b2_span_context_copy vs the reference's ContextSpanCopyLauncher on the
    same contiguous [seq, nG, 128] K rows, span-aligned lengths (the reference quantizes whole spans): every span byte equal."""
    from b200spark import ops
    nH, nG = 8, 2
    cb = ops.SpanCache(1, seq, nH, nG, span, mode)
    ops.context_copy(cb, "k", 0, context_src(mode, span, seq, nG))
    torch.cuda.synchronize()
    assert digest(cb) == _golden()["context_copy"]["mode%d_span%d_seq%d" % (mode, span, seq)]


@pytest.mark.parametrize("mode", [KV.QUANT_NONE, KV.QUANT_I8, KV.QUANT_U4])
def test_context_span_copy_equals_appends_and_handles_ragged_strided_input(mode):
    """A ragged length (not a span multiple) read out of a fused qkv activation (strided rows): the spans equal what
    seq_len single-token appends produce, and the rows past seq_len stay untouched (pool pre-filled with 0xEE)."""
    from b200spark import ops
    nH, nG, span, seq = 8, 2, 32, 77
    width = (nH + 2 * nG) * 128
    rng = np.random.default_rng(5 + mode)
    qkv = torch.from_numpy(rng.standard_normal((seq, width)).astype(np.float32)).to(torch.bfloat16).cuda()
    ca = ops.SpanCache(1, 128, nH, nG, span, mode, fill=0xEE)
    cc = ops.SpanCache(1, 128, nH, nG, span, mode, fill=0xEE)
    pos = torch.zeros(1, dtype=torch.int32, device="cuda")
    for t in range(seq):
        ops.cache_append(ca, qkv[t:t + 1], pos)
        pos += 1
    ops.context_copy(cc, "k", 0, qkv[:, nH * 128:(nH + nG) * 128])
    ops.context_copy(cc, "v", 0, qkv[:, (nH + nG) * 128:])
    torch.cuda.synchronize()
    assert torch.equal(ca.k_pool, cc.k_pool) and torch.equal(ca.v_pool, cc.v_pool)
