"""GPU parity: NeoX rotary embedding at the positions real decoding reaches (up to 32767), in the fused cache append
(head 128 and head 64), the standalone b2_rotary, and the K rows the append stores in NONE / I8 / U4 caches.

Reference: fp64 NeoX rotate-half, inv_i = base^(-2i/d), theta = pos * inv_i.  The kernels compute the angle in fp32
(pos * exp2f(-log2(base) * 2i/d)), so their error grows with the position; bound per element:
    |got - ref| <= 4e-7 * pos * hypot(a, b) + ulp_FT(|ref|)
with (a, b) the rotated input pair: the first term covers the rounding of log2(base), the exponent product, exp2f, the
angle product and sincosf; the second the rounding of the result to the 16-bit type."""
import numpy as np
import pytest
import torch

from oracle import kvcache_ref as KV

pytestmark = pytest.mark.gpu

POSITIONS = [0, 1, 2047, 2048, 4099, 32767]
BASES = [1e4, 5e5, 1e6]
REPS = 4  # sequences per position
NH, NG = 8, 2


def _positions():
    return np.repeat(np.asarray(POSITIONS, np.int64), REPS)


def _ulp(x, dtype):
    m = 7 if dtype == torch.bfloat16 else 10
    return 2.0 ** (np.floor(np.log2(np.maximum(np.abs(x), 2.0 ** -14))) - m)


def _rope_ref(x, pos, base, rdim):
    """x fp64 [B, heads, D], pos [B] -> (rotated fp64, hypot of each element's rotated pair)"""
    half = rdim // 2
    inv = float(base) ** (-np.arange(half, dtype=np.float64) * 2.0 / rdim)
    th = pos.astype(np.float64)[:, None, None] * inv[None, None, :]
    cs, sn = np.cos(th), np.sin(th)
    a, b = x[..., :half], x[..., half:rdim]
    out = x.copy()
    out[..., :half] = a * cs - b * sn
    out[..., half:rdim] = b * cs + a * sn
    hyp = np.zeros_like(x)
    hyp[..., :half] = hyp[..., half:rdim] = np.hypot(a, b)
    return out, hyp


def _check_rope(got, x, pos, base, rdim, dtype, what):
    """got / x: fp32 [B, heads, D] (x = the kernel's input); dims >= rdim must be untouched"""
    ref, hyp = _rope_ref(x.astype(np.float64), pos, base, rdim)
    assert np.array_equal(got[..., rdim:], x[..., rdim:]), (what, "dims past rotary_dim changed")
    err = np.abs(got[..., :rdim] - ref[..., :rdim])
    bound = 4e-7 * pos[:, None, None] * hyp[..., :rdim] + _ulp(ref[..., :rdim], dtype)
    line = " ".join(f"{p}:{err[pos == p].max():.2e}" for p in POSITIONS)
    print(f"\n{what} base {base:g} rotary_dim {rdim} {str(dtype)[6:]}: max |err| per position  {line}")
    bad = err > bound
    assert not bad.any(), (what, pos[np.nonzero(bad)[0][0]], float(err[bad].max()), float(bound[bad][0]))


def _ft_rows(u8, dtype):
    """raw 16-bit cache bytes -> fp32"""
    u16 = u8.view(np.uint16)
    return KV.bits_to_f32(u16) if dtype == torch.bfloat16 else u16.view(np.float16).astype(np.float32)


def _cache_rows(cache, which, pos, head, n_rows_fn):
    """[B, nG, head] rows at each sequence's position, as raw span bytes per (b, g) -> list of uint8 arrays via n_rows_fn"""
    out = []
    S = cache.cfg.span_len
    for b, p in enumerate(pos):
        span = cache.span_view(which, b, int(p) // S).cpu().numpy()
        out.append(n_rows_fn(span, int(p) % S))
    return out


def _none_rows(cache, which, pos, dtype, head=128):
    G, S = cache.cfg.n_groups, cache.cfg.span_len
    rows = _cache_rows(cache, which, pos, head, lambda sp, r: sp[:G * S * head * 2].reshape(G, S, head * 2)[:, r].copy())
    return np.stack([_ft_rows(r, dtype) for r in rows])


def _quant_rows(cache, which, pos, mode):
    G, S = cache.cfg.n_groups, cache.cfg.span_len
    row = {KV.QUANT_I8: 128, KV.QUANT_U4: 64}[mode]

    def get(sp, r):
        d = sp[:G * S * row].reshape(G, S, row)[:, r]
        if mode == KV.QUANT_I8:
            codes = d.view(np.int8).astype(np.int32)
        else:
            codes = np.stack([d & 0xF, d >> 4], -1).reshape(G, 128).astype(np.int32)
        prm = sp[G * S * row:G * S * row + G * S * 8].view(np.float32).reshape(G, S, 2)[:, r]
        return codes, prm
    got = _cache_rows(cache, which, pos, 128, get)
    return np.stack([c for c, _ in got]), np.stack([p for _, p in got])


def _check_quant(codes, prm, x, mode, what):
    """Stored codes / {zero, scale} of rows x [B, nG, 128] against KV.quant_rows (IEEE reciprocal where the kernel uses
    MUFU.RCP): scales identical; a zero point may differ (by 1) only on rows whose zero point is within 1e-4 of a .5 tie;
    codes differ (by 1) only at values within 2e-4 of a .5 tie, or (by <= 2) on a row whose zero point differs."""
    q, z, s = KV.quant_rows(x, mode)
    q = q.astype(np.int32)
    assert np.array_equal(prm[..., 1], s), (what, "scales")
    origin = -128.0 if mode == KV.QUANT_I8 else 0.0
    r = (np.float32(1) / s).astype(np.float64)
    zf = -x.min(-1).astype(np.float64) * r + origin
    ztie = np.abs(zf - np.floor(zf) - 0.5) < 1e-4
    dz = np.abs(prm[..., 0] - z)
    assert dz.max() <= 1 and not (dz[~ztie] != 0).any(), (what, "zero points")
    tf = x.astype(np.float64) * r[..., None] + z[..., None].astype(np.float64)
    ctie = np.abs(tf - np.floor(tf) - 0.5) < 2e-4
    dc = np.abs(codes - q)
    same = (dz == 0)[..., None] & np.ones_like(dc, bool)
    assert dc.max() <= 2 and not (dc[same & ~ctie] != 0).any() and dc[same].max(initial=0) <= 1, (what, "codes")
    return int((dz != 0).sum()), int((dc[same] != 0).sum())


def _append(mode, dtype, qkv, pos, rope, head=128, nH=NH, nG=NG, span=128):
    from b200spark import ops
    B = qkv.shape[0]
    cache = ops.SpanCache(B, max(POSITIONS) + 1, nH, nG, span, mode, dtype=dtype, head=head)
    q = ops.cache_append(cache, qkv.cuda(), torch.from_numpy(pos.astype(np.int32)).cuda(), rope=rope)
    torch.cuda.synchronize()
    return cache, q.float().cpu().numpy().reshape(B, nH, head)


@pytest.mark.parametrize("base", BASES)
@pytest.mark.parametrize("rdim", [128, 64])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_fused_append_rope(dtype, rdim, base):
    """b2_span_cache_append with fused rotary, head 128: q_out and the K row stored in a NONE cache against the fp64
    rotation, the V row bit for bit; the same append into I8 / U4 caches stores exactly the quantization of that K row."""
    pos = _positions()
    B = len(pos)
    g = torch.Generator().manual_seed(int(base) % 1000 + rdim + (1 if dtype == torch.float16 else 0))
    qkv = torch.randn(B, (NH + 2 * NG) * 128, generator=g).to(dtype)
    x = qkv.float().numpy().reshape(B, NH + 2 * NG, 128)
    cache, q = _append(KV.QUANT_NONE, dtype, qkv, pos, (base, rdim))
    _check_rope(q, x[:, :NH], pos, base, rdim, dtype, "fused q_out")
    k = _none_rows(cache, "k", pos, dtype)
    _check_rope(k, x[:, NH:NH + NG], pos, base, rdim, dtype, "fused cached K")
    v = _none_rows(cache, "v", pos, dtype)
    assert np.array_equal(v, x[:, NH + NG:]), "V rows are stored unrotated, bit for bit"
    for mode in (KV.QUANT_I8, KV.QUANT_U4):
        qc, _ = _append(mode, dtype, qkv, pos, (base, rdim))
        for which, rows in (("k", k), ("v", x[:, NH + NG:])):
            codes, prm = _quant_rows(qc, which, pos, mode)
            nz, nc = _check_quant(codes, prm, rows, mode, (mode, which))
            print(f"  mode {mode} {which}: zero-point ties {nz}, code ties {nc}")


@pytest.mark.parametrize("base", BASES)
@pytest.mark.parametrize("rdim", [128, 64])
def test_standalone_rotary(rdim, base):
    """b2_rotary (in place on a fused qkv row, bf16): q and k heads against the fp64 rotation, V untouched, and within one
    bf16 ulp of the fused append's q_out / cached K — the two evaluate the same formula."""
    from b200spark import ops
    pos = _positions()
    B = len(pos)
    g = torch.Generator().manual_seed(int(base) % 997 + rdim)
    qkv = torch.randn(B, (NH + 2 * NG) * 128, generator=g).to(torch.bfloat16)
    x = qkv.float().numpy().reshape(B, NH + 2 * NG, 128)
    r = ops.rotary(qkv.cuda(), torch.from_numpy(pos.astype(np.int32)).cuda(), NH, NG, base=base, rotary_dim=rdim)
    torch.cuda.synchronize()
    got = r.float().cpu().numpy().reshape(B, NH + 2 * NG, 128)
    _check_rope(got[:, :NH + NG], x[:, :NH + NG], pos, base, rdim, torch.bfloat16, "b2_rotary")
    assert np.array_equal(got[:, NH + NG:], x[:, NH + NG:])
    cache, q = _append(KV.QUANT_NONE, torch.bfloat16, qkv, pos, (base, rdim))
    fused = np.concatenate([q, _none_rows(cache, "k", pos, torch.bfloat16)], 1)
    d = np.abs(fused - got[:, :NH + NG])
    assert np.all(d <= _ulp(np.maximum(np.abs(fused), np.abs(got[:, :NH + NG])), torch.bfloat16)), float(d.max())


@pytest.mark.parametrize("base", BASES)
@pytest.mark.parametrize("rdim", [64, 32])
def test_head64_append_rope(rdim, base):
    """cache_append64_kernel (bf16, head 64): q_out and the cached K row against the fp64 rotation, V bit for bit"""
    nH, nG = 14, 2
    pos = _positions()
    B = len(pos)
    g = torch.Generator().manual_seed(int(base) % 991 + rdim)
    qkv = torch.randn(B, (nH + 2 * nG) * 64, generator=g).to(torch.bfloat16)
    x = qkv.float().numpy().reshape(B, nH + 2 * nG, 64)
    cache, q = _append(KV.QUANT_NONE, torch.bfloat16, qkv, pos, (base, rdim), head=64, nH=nH, nG=nG)
    _check_rope(q, x[:, :nH], pos, base, rdim, torch.bfloat16, "head-64 q_out")
    k = _none_rows(cache, "k", pos, torch.bfloat16, head=64)
    _check_rope(k, x[:, nH:nH + nG], pos, base, rdim, torch.bfloat16, "head-64 cached K")
    assert np.array_equal(_none_rows(cache, "v", pos, torch.bfloat16, head=64), x[:, nH + nG:])
