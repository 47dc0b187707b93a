"""GPU parity: span attention at the work schedules the decode step really runs, and the head-64 kernels.

span_attn_kernel cuts the flat list of (sequence, kv-head, 64-token tile) into equal ranges of Tc tiles, one range per CTA of a
persistent grid (occupancy x SMs).  At the benchmark's launch (Qwen2-7B, batch 64, ctx 2048) a CTA streams ~20 tiles through
its cp.async ring and covers the tail of one (sequence, kv-head) and the head of the next; a ragged batch puts whole short
(sequence, kv-head)s between two partial pieces.  `_schedule` restates the decomposition so that every case asserts the
regime it claims to reach.  The grid is read back from the handle (its workspace holds two partial slots per CTA).

Every oracle comparison attends over the device's own cache bytes (pools read back through the page permutation)."""
import bisect
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import kvcache_ref as KV

NH, NG, SPAN = 28, 4, 128  # Qwen2-7B attention geometry
TILE = 64
DEFAULT_STAGES = {KV.QUANT_NONE: 2, KV.QUANT_I8: 3, KV.QUANT_U4: 4}
RAGGED_CHOICES = [1, 17, 64, 65, 200, 777, 2049, 4100]
B2_ERR_LIMIT, B2_ERR_UNSUPPORTED = 4, 6


# ---------------------------------------------------------------------------------------------------------------------
# schedule model (span_attn.cu, span_attn_kernel: "device-side work decomposition" and "locate (b, g, first tile)")
# ---------------------------------------------------------------------------------------------------------------------
def _schedule(lens, n_groups, grid, max_pieces=1 << 20):
    """-> (Tc, per-CTA list of pieces (b, g, t0, ntiles, npieces))"""
    tiles = [(int(n) + TILE - 1) // TILE for n in lens]
    total = sum(tiles) * n_groups
    Tc = max(-(-total // grid), -(-max(tiles) // max_pieces), 1)
    prefix = np.concatenate([[0], np.cumsum(np.asarray(tiles) * n_groups)]).tolist()
    ctas = []
    for c in range(grid):
        lo, hi = c * Tc, min(total, c * Tc + Tc)
        pieces, pos = [], lo
        while pos < hi:
            b = bisect.bisect_right(prefix, pos, 0, len(tiles)) - 1
            within = pos - prefix[b]
            g, t0 = divmod(within, tiles[b])
            bg_start = prefix[b] + g * tiles[b]
            bg_end = bg_start + tiles[b]
            pend = min(hi, bg_end)
            pieces.append((b, g, t0, pend - pos, (bg_end - 1) // Tc - bg_start // Tc + 1))
            pos = pend
        ctas.append(pieces)
    return Tc, ctas


def _whole_between_partials(ctas):
    """CTAs whose range holds a whole (sequence, kv-head) (direct write) between two split pieces"""
    return sum(1 for ps in ctas if len(ps) >= 3 and ps[0][4] > 1 and ps[-1][4] > 1 and any(p[4] == 1 for p in ps[1:-1]))


def _max_piece(ctas):
    return max((p[3] for ps in ctas for p in ps), default=0)


def _max_npieces(ctas):
    return max((p[4] for ps in ctas for p in ps), default=0)


def _grid_of(attn, B, max_len):
    """b2_span_attn_workspace_bytes = 2 levels x (2 slots per CTA) x hpg x (128 + 2) fp32 + 256"""
    hpg = attn.cfg.n_heads // attn.cfg.n_groups
    ws = attn.workspace_bytes(B, max_len) - 256
    assert ws % (16 * hpg * 130) == 0
    return ws // (16 * hpg * 130)


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------
# cache fill (prefill span writer) and oracle read-back
# ---------------------------------------------------------------------------------------------------------------------
def _fill(mode, lens, nH, nG, span, seed, dtype=torch.bfloat16, max_len=None):
    """Sequence b's K and V rows (seeded N(0,1) in `dtype`) written by b2_span_context_copy; q [B, nH*128] alike."""
    from b200spark import ops
    B = len(lens)
    max_len = max_len or max(lens)
    cache = ops.SpanCache(B, max_len, nH, nG, span, mode, dtype=dtype)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    for b in range(B):
        rows = torch.randn(int(lens[b]), 2 * nG * 128, generator=gen, device="cuda").to(dtype)
        ops.context_copy(cache, "k", b, rows[:, :nG * 128])
        ops.context_copy(cache, "v", b, rows[:, nG * 128:])
    q = torch.randn(B, nH * 128, generator=gen, device="cuda").to(dtype)
    torch.cuda.synchronize()
    return cache, q


def _oracle_caches(cache, lens):
    """SpanCacheRef views of the device's K and V pools: ONE device-to-host copy per pool, sliced through the page tables."""
    cfg = cache.cfg
    ft = "fp16" if cache.dtype == torch.float16 else "bf16"
    out = []
    for pool, perm in ((cache.k_pool, cache.perm_k), (cache.v_pool, cache.perm_v)):
        host = pool.cpu().numpy().reshape(-1, cache.stride)
        ref = KV.SpanCacheRef(cfg.quant_mode, cfg.span_len, cfg.n_groups, head=cache.head, ft=ft)
        for b, n in enumerate(lens):
            ref.spans.append([host[int(perm[b, si]), :cache.span_bytes] for si in range(-(-int(n) // cfg.span_len))])
        out.append(ref)
    return out


def _reference(cache, q, lens):
    kref, vref = _oracle_caches(cache, lens)
    nH, hd = cache.cfg.n_heads, cache.head
    return KV.attention_ref(q.float().cpu().numpy().reshape(len(lens), nH, hd), kref, vref, list(lens), nH, 1.0 / np.sqrt(hd))


def _weighted_abs_v(cache, q, lens):
    """S[b, h, d] = sum_j p_j |V_j[d]| in fp64 (p = the oracle's softmax): the scale of an error made on the probabilities"""
    kref, vref = _oracle_caches(cache, lens)
    nH, hd, G = cache.cfg.n_heads, cache.head, cache.cfg.n_groups
    qf = q.float().cpu().numpy().reshape(len(lens), nH, hd).astype(np.float64)
    S = np.zeros((len(lens), nH, hd))
    for b, n in enumerate(lens):
        K, V = kref.dense(b, int(n)).astype(np.float64), np.abs(vref.dense(b, int(n)).astype(np.float64))
        for h in range(nH):
            s = K[h // (nH // G)] @ qf[b, h] / np.sqrt(hd)
            pr = np.exp(s - s.max())
            S[b, h] = pr @ V[h // (nH // G)] / pr.sum()
    return S


def _check_oracle(got, ref, mode, dtype):
    """tests/test_attn_gpu.py's bounds for the same mode and type.  bf16 NONE: its 6e-3 absolute bound holds for outputs up
    to ~1 (long sequences); a short sequence averages a few N(0,1) rows and its outputs reach ~3, where the bf16 rounding of
    the output and of the probabilities alone is 2^-9 |out| each, so the bound carries 2^-8 |ref| on top."""
    err = np.abs(got - ref)
    if mode == KV.QUANT_NONE and dtype == torch.float16:
        bound = 2e-3 + 2.0 ** -9 * np.abs(ref)
    elif mode == KV.QUANT_NONE:
        bound = 6e-3 + 2.0 ** -8 * np.abs(ref)
    else:
        bound = 2e-3 + 2.0 ** -7 * np.abs(ref)
    i = np.unravel_index(np.argmax(err), err.shape)
    return bool(np.all(err <= bound)), f"max |out - oracle| {float(err[i]):.3e} at |ref| {float(np.abs(ref[i])):.3f}"


def _ulp(x, dtype):
    m = 7 if dtype == torch.bfloat16 else 10
    return 2.0 ** (np.floor(np.log2(np.maximum(np.abs(x), 2.0 ** -14))) - m)


def _run_attn(attn, cache, q, lens, max_len):
    from b200spark import ops
    new_lens = torch.tensor([int(n) for n in lens], dtype=torch.int32, device="cuda")
    out = attn(q, cache, new_lens, max_len, ops.Workspace())
    torch.cuda.synchronize()
    return out


def _handle(monkeypatch, cfg, max_batch, **env):
    from b200spark import ops
    for k in ("B2_ATTN_STAGES", "B2_ATTN_CTAS_PER_SM", "B2_ATTN_MAX_PIECES"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    return ops.SpanAttn(cfg, max_batch)


MODES = [(KV.QUANT_NONE, torch.bfloat16), (KV.QUANT_I8, torch.bfloat16), (KV.QUANT_U4, torch.bfloat16),
         (KV.QUANT_NONE, torch.float16), (KV.QUANT_I8, torch.float16)]
MODE_IDS = ["none-bf16", "i8-bf16", "u4-bf16", "none-fp16", "i8-fp16"]


def test_schedule_model_known_answers():
    """The schedule model by hand (no device needed): bench.py's launch at 444 CTAs takes Tc = 20 and puts the
    end of one (sequence, kv-head) and the start of the next into one CTA; a single long sequence is split evenly."""
    Tc, ctas = _schedule([2049] * 64, 4, 444)
    assert Tc == 20 and _max_piece(ctas) == 20 and sum(len(ps) for ps in ctas) > 444
    assert sum(p[3] for ps in ctas for p in ps) == 64 * 4 * 33
    Tc, ctas = _schedule([2048], 4, 148, max_pieces=4)
    assert Tc == 8 and _max_npieces(ctas) == 4
    Tc, ctas = _schedule([1, 300, 5000], 2, 7)
    covered = sorted((p[0], p[1], p[2] + i) for ps in ctas for p in ps for i in range(p[3]))
    assert covered == sorted((b, g, t) for b, n in enumerate([1, 300, 5000]) for g in range(2) for t in range(-(-n // 64)))


# ---------------------------------------------------------------------------------------------------------------------
# B1: the benchmark's launch
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode,dtype", MODES, ids=MODE_IDS)
def test_attention_bench_launch(monkeypatch, mode, dtype):
    """B = 64, every length 2049 (bench.py's ctx 2048 + the new token): pieces far longer than the ring, the tail of one
    (sequence, kv-head) and the head of the next in one CTA, the direct last-CTA merge.  Two runs are bit-identical."""
    lens = [2049] * 64
    cache, q = _fill(mode, lens, NH, NG, SPAN, seed=100 + mode + (7 if dtype == torch.float16 else 0), dtype=dtype)
    attn = _handle(monkeypatch, cache.cfg, 64)
    grid = _grid_of(attn, 64, 2049)
    Tc, ctas = _schedule(lens, NG, grid)
    print(f"\nmode {mode} {dtype}: grid {grid}, Tc {Tc}, longest piece {_max_piece(ctas)} tiles, pieces/(seq,head) <= {_max_npieces(ctas)}")
    assert _max_piece(ctas) >= 9, "pieces of more than 8 tiles"
    assert _max_piece(ctas) > DEFAULT_STAGES[mode], "the cp.async ring wraps"
    assert any(len(ps) >= 2 for ps in ctas), "a CTA finishes one (sequence, kv-head) and starts the next"
    out = _run_attn(attn, cache, q, lens, 2049)
    out2 = _run_attn(attn, cache, q, lens, 2049)
    assert torch.equal(out, out2)
    ok, err = _check_oracle(out.float().cpu().numpy().reshape(64, NH, 128), _reference(cache, q, lens), mode, dtype)
    print("  " + err)
    assert ok, err


# ---------------------------------------------------------------------------------------------------------------------
# B2 + B3: a ragged serving batch, and the same cache under every schedule knob
# ---------------------------------------------------------------------------------------------------------------------
def _ragged_lens(seed=2024):
    return [int(n) for n in np.random.default_rng(seed).choice(RAGGED_CHOICES, size=64)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,dtype", MODES, ids=MODE_IDS)
def test_attention_ragged_all_schedules(monkeypatch, mode, dtype):
    """B = 64 with lengths from {1, 17, 64, 65, 200, 777, 2049, 4100}.  One CTA per SM: some CTA's range holds a whole
    (sequence, kv-head) between two split pieces.  The same cache is then attended under the default handle, one CTA per
    SM, 2 / 3 / 4 ring stages and at most 4 pieces per (sequence, kv-head): every result within the oracle bound, and all
    within 1e-5 + 1 ulp of each other (only the fp32 summation order differs)."""
    lens = _ragged_lens()
    assert set(lens) == set(RAGGED_CHOICES)
    L = max(lens)
    cache, q = _fill(mode, lens, NH, NG, SPAN, seed=200 + mode + (7 if dtype == torch.float16 else 0), dtype=dtype)
    ref = _reference(cache, q, lens)
    settings = [("default", {}), ("ctas_per_sm=1", {"B2_ATTN_CTAS_PER_SM": 1})] + \
               [(f"stages={s}", {"B2_ATTN_STAGES": s}) for s in (2, 3, 4)] + [("max_pieces=4", {"B2_ATTN_MAX_PIECES": 4})]
    outs, plans = {}, {}
    for name, env in settings:
        attn = _handle(monkeypatch, cache.cfg, 64, **env)
        grid = _grid_of(attn, 64, L)
        Tc, ctas = _schedule(lens, NG, grid, int(env.get("B2_ATTN_MAX_PIECES", 1 << 20)))
        stages = int(env.get("B2_ATTN_STAGES", DEFAULT_STAGES[mode]))
        plans[name] = (grid, Tc, stages, [[p[:4] for p in ps] for ps in ctas])
        outs[name] = _run_attn(attn, cache, q, lens, L)
        got = outs[name].float().cpu().numpy().reshape(64, NH, 128)
        ok, err = _check_oracle(got, ref, mode, dtype)
        print(f"\n{name:14s} grid {grid:4d} Tc {Tc:3d} stages {stages} longest piece {_max_piece(ctas):3d} "
              f"whole-between-partials CTAs {_whole_between_partials(ctas):3d} max pieces {_max_npieces(ctas):3d}: {err}")
        assert ok, (name, err)
        assert _max_piece(ctas) > stages, (name, "the ring wraps")
        if name == "ctas_per_sm=1":
            assert grid == _sm_count(), "one CTA per SM: the grid is the SM count"
            assert _whole_between_partials(ctas) > 0
            assert _max_piece(ctas) > 8 and _max_piece(ctas) > stages
    d_grid, d_Tc, d_st, d_pieces = plans["default"]
    for name, (grid, Tc, stages, pieces) in plans.items():
        if name == "default" or (name.startswith("stages=") and stages == d_st):
            continue  # the default configuration itself
        # a knob must change the schedule (Tc or the piece boundaries) or the ring depth it streams through
        assert (Tc, pieces) != (d_Tc, d_pieces) or stages != d_st, name
        if name == "max_pieces=4":
            assert Tc != d_Tc, "the piece cap binds on this batch"
    # The settings differ by more than fp32 reassociation: the MMA takes the probabilities as 16-bit operands (bf16 for a
    # bf16 NONE cache, fp16 otherwise), exp2(s - m) rounded relative to the running max m of the PIECE, and the piece
    # boundaries move with the schedule.  Each output carries its own rounding of P, <= u_P relative per probability, so
    # two schedules may differ by 2 u_P sum_j p_j |v_j| (P and its row sum) on top of one output rounding each.
    u_p = 2.0 ** -9 if (mode == KV.QUANT_NONE and dtype == torch.bfloat16) else 2.0 ** -11
    S = _weighted_abs_v(cache, q, lens).reshape(64, -1)
    base = outs["default"].float().cpu().numpy().reshape(64, -1)
    worst = 0.0
    for name, o in outs.items():
        o = o.float().cpu().numpy().reshape(64, -1)
        tol = 1e-5 + 2 * _ulp(np.maximum(np.abs(o), np.abs(base)), dtype) + 4 * u_p * S
        r = np.abs(o - base) / tol
        assert r.max() <= 1, (name, float(np.abs(o - base).max()), float(r.max()))
        worst = max(worst, float(r.max()))
    print(f"max |out(setting) - out(default)| / bound over all settings: {worst:.3f}")


# ---------------------------------------------------------------------------------------------------------------------
# B4: batch limits
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", [KV.QUANT_NONE, KV.QUANT_I8, KV.QUANT_U4])
@pytest.mark.parametrize("B", [33, 1000, 1024])
def test_attention_large_batch(monkeypatch, B, mode):
    """Batches above 64 up to kMaxBatch = 1024, short ragged lengths (1..300), (8, 2) heads: the lengths' prefix scan
    over several 32-wide warp passes and the binary search over up to 1024 sequences."""
    nH, nG, span = 8, 2, 64
    lens = np.random.default_rng(B + 10 * mode).integers(1, 301, size=B).tolist()
    cache, q = _fill(mode, lens, nH, nG, span, seed=300 + B + mode, max_len=320)
    attn = _handle(monkeypatch, cache.cfg, B)
    Tc, ctas = _schedule(lens, nG, _grid_of(attn, B, 320))
    assert max(p[0] for ps in ctas for p in ps) == B - 1
    out = _run_attn(attn, cache, q, lens, 320)
    ok, err = _check_oracle(out.float().cpu().numpy().reshape(B, nH, 128), _reference(cache, q, lens), mode, torch.bfloat16)
    print(f"\nB {B} mode {mode}: Tc {Tc}, {err}")
    assert ok, err


@pytest.mark.gpu
def test_attention_batch_limits():
    from b200spark import ops
    from b200spark._lib import lib
    cache = ops.SpanCache(4, 256, 8, 2, 64, KV.QUANT_NONE)
    h = C.c_void_p()
    assert lib.b2_span_attn_create(C.byref(h), C.byref(cache.cfg), 1025) == B2_ERR_LIMIT
    attn = ops.SpanAttn(cache.cfg, 2)
    ws = ops.Workspace()
    wsb = ws.reserve(attn.workspace_bytes(4, 256))
    q = torch.zeros(4, 8 * 128, dtype=torch.bfloat16, device="cuda")
    out = torch.empty_like(q)
    lens = torch.ones(4, dtype=torch.int32, device="cuda")
    st = lib.b2_span_attn_run(attn.h, C.c_void_p(out.data_ptr()), C.c_void_p(q.data_ptr()), C.c_void_p(cache.k_tab.data_ptr()),
                              C.c_void_p(cache.v_tab.data_ptr()), C.c_void_p(lens.data_ptr()), 3, 256, C.c_void_p(wsb.data_ptr()),
                              wsb.numel(), 1.0, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert st == B2_ERR_LIMIT


# ---------------------------------------------------------------------------------------------------------------------
# B5: a decode loop whose schedule shifts under it, eager and as a replayed CUDA graph
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_decode_loop_schedule_shift_graph_replay(monkeypatch):
    """B = 64 from length 2045, six steps of append (fused RoPE, base 1e6) -> attention -> lens_add: the attended lengths
    cross 2048 -> 2049, so the tile count, Tc and the piece boundaries change while the handle's merge counters re-arm.
    A captured step replayed six times gives the eager loop's outputs bit for bit; the last step matches the oracle."""
    from b200spark import ops
    B, L0, steps = 64, 2045, 6
    max_len = L0 + steps + 1
    cache, _ = _fill(KV.QUANT_NONE, [L0] * B, NH, NG, SPAN, seed=500, max_len=max_len)
    attn = _handle(monkeypatch, cache.cfg, B)
    grid = _grid_of(attn, B, max_len)
    plans = [_schedule([L0 + 1 + t] * B, NG, grid) for t in range(steps)]
    for t in range(steps):
        print(f"\nstep {t}: attended length {L0 + 1 + t}, Tc {plans[t][0]}")
    assert len({(Tc, tuple(tuple(p[:4] for p in ps) for ps in c)) for Tc, c in plans}) >= 2, "the schedule changes"
    gen = torch.Generator(device="cuda").manual_seed(501)
    qkv_steps = [torch.randn(B, (NH + 2 * NG) * 128, generator=gen, device="cuda").to(torch.bfloat16) for _ in range(steps)]
    ws = ops.Workspace()
    ws.reserve(attn.workspace_bytes(B, max_len))
    lens_old = torch.full((B,), L0, dtype=torch.int32, device="cuda")
    lens_new = lens_old + 1
    qkv = torch.empty_like(qkv_steps[0])
    q = torch.empty(B, NH * 128, dtype=torch.bfloat16, device="cuda")
    out = torch.empty_like(q)

    def step():
        ops.cache_append(cache, qkv, lens_old, q_out=q, rope=(1e6, 128))
        attn(q, cache, lens_new, max_len, ws, out=out)
        ops.lens_add(lens_old, 1)
        ops.lens_add(lens_new, 1)

    eager = []
    for t in range(steps):
        qkv.copy_(qkv_steps[t])
        step()
        eager.append(out.clone())
    torch.cuda.synchronize()
    q_last = q.clone()
    lens_old.fill_(L0); lens_new.fill_(L0 + 1)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    torch.cuda.synchronize()
    lens_old.fill_(L0); lens_new.fill_(L0 + 1)  # capture does not execute, but keep the start state explicit
    for t in range(steps):
        qkv.copy_(qkv_steps[t])
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager[t]), t
    assert lens_old.cpu().tolist() == [L0 + steps] * B
    assert torch.equal(q, q_last)
    lens = [L0 + steps] * B
    ok, err = _check_oracle(eager[-1].float().cpu().numpy().reshape(B, NH, 128), _reference(cache, q_last, lens),
                            KV.QUANT_NONE, torch.bfloat16)
    print(f"last step: {err}")
    assert ok, err


# ---------------------------------------------------------------------------------------------------------------------
# D: the head-64 kernels (span_attn64.cu), bf16 KV
# ---------------------------------------------------------------------------------------------------------------------
def _fill64(lens, nH, nG, span, seed, fill=0):
    """Head-64 K / V rows written straight into the span pages ([nG][span][64] bf16 per page) with torch; rows past each
    length keep the pool's fill byte."""
    from b200spark import ops
    B = len(lens)
    cache = ops.SpanCache(B, max(lens), nH, nG, span, KV.QUANT_NONE, head=64, fill=fill)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    for pool, perm in ((cache.k_pool, cache.perm_k), (cache.v_pool, cache.perm_v)):
        pages = pool.view(-1, cache.stride)
        for b, n in enumerate(lens):
            rows = torch.randn(n, nG, 64, generator=gen, device="cuda").to(torch.bfloat16)
            for si in range(-(-n // span)):
                k = min(span, n - si * span)
                page = pages[int(perm[b, si]), :cache.span_bytes].view(torch.bfloat16).view(nG, span, 64)
                page[:, :k] = rows[si * span: si * span + k].transpose(0, 1)
    q = torch.randn(B, nH * 64, generator=gen, device="cuda").to(torch.bfloat16)
    torch.cuda.synchronize()
    return cache, q


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 5, 64])
@pytest.mark.parametrize("nH,nG", [(14, 2), (16, 1), (8, 8), (12, 4)])
@pytest.mark.parametrize("span", [16, 32, 64, 128])
def test_attention_head64(span, nH, nG, B):
    from b200spark import ops
    rng = np.random.default_rng(span * 100 + nH * 10 + nG + B)
    lens = [2049] if B == 1 else rng.integers(1, 2050, size=B).tolist()
    if B > 1:
        lens[0], lens[1] = 1, 2049
    cache, q = _fill64(lens, nH, nG, span, seed=600 + span + nH + B)
    out = _run_attn(ops.SpanAttn(cache.cfg, B), cache, q, lens, max(lens))
    ok, err = _check_oracle(out.float().cpu().numpy().reshape(B, nH, 64), _reference(cache, q, lens), KV.QUANT_NONE, torch.bfloat16)
    print(f"\nhead 64, span {span}, ({nH}, {nG}), B {B}: {err}")
    assert ok, err


@pytest.mark.gpu
@pytest.mark.parametrize("span", [16, 128])
def test_attention_head64_unwritten_memory(span):
    """0xFF-filled pools (NaN as bf16): only rows below each length may reach the output"""
    from b200spark import ops
    lens = [1, 37, 129, 191, 1000]
    cache, q = _fill64(lens, 14, 2, span, seed=700 + span, fill=0xFF)
    out = _run_attn(ops.SpanAttn(cache.cfg, len(lens)), cache, q, lens, max(lens))
    got = out.float().cpu().numpy().reshape(len(lens), 14, 64)
    assert np.isfinite(got).all()
    ok, err = _check_oracle(got, _reference(cache, q, lens), KV.QUANT_NONE, torch.bfloat16)
    assert ok, err


@pytest.mark.gpu
@pytest.mark.parametrize("mode,dtype", [(KV.QUANT_I8, torch.bfloat16), (KV.QUANT_U4, torch.bfloat16), (KV.QUANT_NONE, torch.float16)])
def test_head64_rejects_other_cache_types(mode, dtype):
    from b200spark._lib import DT_BF16, DT_F16, SpanCfg, lib
    cfg = SpanCfg(DT_F16 if dtype == torch.float16 else DT_BF16, mode, 14, 2, 64, 16, 8, 0)
    h = C.c_void_p()
    assert lib.b2_span_attn_create(C.byref(h), C.byref(cfg), 4) == B2_ERR_UNSUPPORTED
    assert lib.b2_span_bytes(C.byref(cfg)) == 0


# ---------------------------------------------------------------------------------------------------------------------
# E: the benchmark's decode step end to end at its real context, at the three batches bench.py reports
# ---------------------------------------------------------------------------------------------------------------------
def _seed_oracle(ref, st, b):
    """RefDecoder's per-layer K / V row lists <- the first b sequences' cached rows (device bytes)"""
    n = int(st.lens_old[0].item())
    ref.reset(b)
    for li, L in enumerate(st.layers):
        kref, vref = _oracle_caches(L["cache"], [n] * st.Bmax)
        for s in range(b):
            ref.k[li][s] = list(torch.from_numpy(kref.dense(s, n)).unbind(1))
            ref.v[li][s] = list(torch.from_numpy(vref.dense(s, n)).unbind(1))


@pytest.mark.gpu
def test_bench_step_at_context_2048():
    """One full-width Qwen2-7B layer (int4 per-channel) + lm_head at ctx 2048, span 128: two steps at batch 64, then — on the
    same stack, lengths rewound — at batch 8 and batch 1, the launches bench.py times, with RoPE at position 2048 and up;
    logits and greedy tokens against the reference-CPU-path oracle as in test_full_width_qwen2_7b_layer_and_lm_head."""
    from b200spark import model
    from oracle import decoder_ref as DR
    ctx, steps = 2048, 2
    st = model.DecodeStack(model.QWEN2_7B, 64, ctx + 8, wbits=4, kv="none", span=128, layers=1, keep_ref=True)
    st.set_context(ctx)
    ref = DR.from_stack(st, KV.QUANT_NONE)
    grid = _grid_of(st.attn, 64, ctx + 8)
    for b in (64, 8, 1):
        st._lens_old.fill_(ctx); st._lens_new.fill_(ctx + 1)
        st.set_batch(b)
        Tc, ctas = _schedule([ctx + 1] * b, model.QWEN2_7B.n_kv, grid)
        print(f"\nbatch {b}: Tc {Tc}, pieces per (seq, kv-head) <= {_max_npieces(ctas)}")
        if b == 1:
            assert _max_npieces(ctas) > 16, "two-level merge"
        _seed_oracle(ref, st, b)
        ids = torch.randint(0, model.QWEN2_7B.vocab, (b,), generator=torch.Generator().manual_seed(4321 + b), dtype=torch.int64)
        for t in range(steps):
            st.ids.copy_(ids.cuda())
            nxt = st.step().cpu()
            torch.cuda.synchronize()
            glog = st.logits.float().cpu()
            rlog, rnext = ref.step(ids, [ctx + t] * b)
            mx = rlog.abs().max().item()
            tol = 1e-2 * mx + 2.0 ** (np.floor(np.log2(mx)) - 7)
            err = (glog - rlog).abs().max().item()
            print(f"  step {t}: max |logit err| {err:.3e} (tol {tol:.3e})")
            assert err <= tol, (b, t, err, tol)
            assert torch.equal(nxt, torch.argmax(glog, dim=-1))
            top2 = torch.topk(rlog, 2, dim=-1).values
            for s in range(b):
                if (top2[s, 0] - top2[s, 1]).item() > 2 * tol:
                    assert nxt[s].item() == rnext[s].item(), (b, t, s)
            ids = nxt
        assert st.lens_old.cpu().tolist() == [ctx + steps] * b
