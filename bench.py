#!/usr/bin/env python
"""bench.py — decode tokens/s of Qwen2-7B IQ-int4 (BASELINE.json configs[1]) through the b200spark C ABI.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W   (the reference's CPU path, restated; rank 0 only)
  python bench.py ... --dump-outputs DIR   (also writes the last timed step's next_ids / logits: dump_outputs())

A "step" is one decode step of the full 28-layer stack + lm_head + greedy sampling for a batch of B sequences at
context ctx, replayed from a CUDA graph.  Prints ONE JSON line (see DESIGN.md "Measurement"):

  value / e2e / roofline / kernels   the headline batch (default 64: configs[1]'s largest batch)
  batches                            the metric's other batches ("b=1..64": 8 and 1) on the SAME weights and caches:
                                     tokens/s, e2e, step fraction of the HBM roofline, per-kernel fractions
  tp  (torchrun, N > 1 only)         config C4: ONE Qwen2-72B int4 instance tensor-parallel over the N ranks, batch 16,
                                     ctx 4096: tokens/s, per-rank roofline fraction, share of the step in the collective
  cpu_baseline (N = 1 only)          the reference's CPU path (restated), bounded sample, on this box's host cores

With N > 1 the headline numbers are N independent replicas of the one-GPU workload (Qwen2-7B fits one GPU: weak scaling,
no data-path collective); the `tp` record is the design's real multi-GPU path.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "dash-infer_b200", "python"))

METRIC = "decode tokens/sec/GPU Qwen2-7B int4-IQ b=1..64; HBM GB/s vs roofline"

# plain dims (SURVEY.md §8): the reference arm must not import the product package (it would map libb200spark.so)
MODEL_DIMS = {
    "qwen2-7b": dict(name="Qwen2-7B", hidden=3584, n_heads=28, n_kv=4, inter=18944, layers=28, vocab=152064, eps=1e-6),
    "llama3-8b": dict(name="Llama-3-8B", hidden=4096, n_heads=32, n_kv=8, inter=14336, layers=32, vocab=128256, eps=1e-5),
    "qwen2-72b": dict(name="Qwen2-72B", hidden=8192, n_heads=64, n_kv=8, inter=29568, layers=80, vocab=152064, eps=1e-6),
    "tiny": dict(name="tiny-2L", hidden=512, n_heads=8, n_kv=2, inter=1024, layers=2, vocab=1024, eps=1e-6),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def physical_cores():
    """Distinct (socket, core) pairs: the thread count torch picks by default outside torchrun (one per physical core).
    torchrun exports OMP_NUM_THREADS=1, so the CPU legs set the pool size explicitly."""
    try:
        seen, phys = set(), None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                seen.add((phys, line.split(":")[1].strip()))
        if seen:
            return len(seen)
    except OSError:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def time_kernel_loop(fn_list, rounds, torch):
    """Average device time per launch over len(fn_list)*rounds launches replayed from a CUDA graph (CUDA events on the
    replaying stream; a graph keeps the host's per-call ctypes overhead out of the measurement, exactly like the decode
    step).  fn_list cycles through DIFFERENT layers' weights/caches so every launch reads fresh HBM (>> L2)."""
    for f in fn_list:
        f()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(rounds):
            for f in fn_list:
                f()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / (rounds * len(fn_list))


def rewind(st, ctx):
    """Sequence lengths back to `ctx` (rows beyond it hold older tokens and are overwritten again)."""
    st._lens_old.fill_(ctx)
    st._lens_new.fill_(ctx + 1)


def timed_steps(st, K, W, torch, dist, world, sampler=None):
    """W untimed + K timed graph replays, barrier + synchronize on both sides, CUDA events, max over ranks -> ms."""
    for _ in range(W):
        st.step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        st.step()           # next_ids stay on device; ids of step t+1 are synthetic (no data dependence on sampling)
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler is not None else None
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, clocks


def e2e_steps(st, ids, K, torch, dist, world):
    """The same step through the public API with HOST buffers: pinned H2D of the ids, D2H of the sampled ids, stream sync
    (a serving loop needs the token on the host before the next step) — wall clock, max over ranks."""
    B = st.B
    ids_host = ids[:B].clone().pin_memory()
    out_host = torch.empty(B, dtype=torch.int64).pin_memory()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        st.ids.copy_(ids_host, non_blocking=True)
        st.step()
        out_host.copy_(st.next_ids, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        ids_host.copy_(out_host)
    s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([s], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        s = float(t.item())
    return s


def kernel_rooflines(st, cfg, hbm_peak, torch, traffic):
    """Per-kernel achieved HBM GB/s at the stack's CURRENT batch, measured live with CUDA events (each launch reads a
    different layer's weights / cache: >> L2)."""
    B, ws, xn = st.B, st.ws, st.xn
    nl = len(st.layers)
    rounds = max(2, 112 // max(1, nl))
    kern = {}
    io = {"gate": (xn, st.gate), "gateup": (xn, st.gate), "up": (xn, st.up), "qkv": (xn, st.qkv), "o": (st.ao, st.x),
          "down": (st.gate, st.x)}

    def entry(name, t, nb, per_step, tkey, note=None):
        e = {"us": round(t * 1e6, 2), "GBps": round(nb / t / 1e9, 1), "frac": round(nb / t / 1e9 / hbm_peak, 3),
             "algo_bytes": nb, "launches_per_step": per_step, "traffic": traffic.get("%s B=%d" % (tkey, B))}
        if note:
            e["note"] = note
        kern[name] = e

    def gemm_entry(name, key, tkey, act=0):
        src, dst = io[key]
        fns = [(lambda L=L: L[key](src, ws, out=dst, act=act)) for L in st.layers]
        t = time_kernel_loop(fns, rounds, torch)
        entry(name, t, st.layers[0][key].op.algo_bytes(B), nl, tkey)

    from b200spark._lib import ACT_SILU
    if st.fuse_swiglu:
        gemm_entry("wq_gemm[gate+up SwiGLU %dx2x%d]" % (cfg.hidden, cfg.inter), "gateup", "wq_gemm[gate+up]")
    else:
        gemm_entry("wq_gemm[gate %dx%d]" % (cfg.hidden, cfg.inter), "gate", "wq_gemm[gate]", ACT_SILU)
        gemm_entry("wq_gemm[up %dx%d]" % (cfg.hidden, cfg.inter), "up", "wq_gemm[up]")
    gemm_entry("wq_gemm[down %dx%d]" % (cfg.inter, cfg.hidden), "down", "wq_gemm[down]")
    gemm_entry("wq_gemm[qkv %dx%d]" % (cfg.hidden, (cfg.n_heads + 2 * cfg.n_kv) * 128), "qkv", "wq_gemm[qkv]")
    gemm_entry("wq_gemm[o %dx%d]" % (cfg.n_heads * 128, cfg.hidden), "o", "wq_gemm[o]")
    cur = int(st.lens_new[0].item())
    fns = [(lambda L=L: st.attn(st.q, L["cache"], st.lens_new, st.max_len, ws, out=st.ao)) for L in st.layers]
    t = time_kernel_loop(fns, rounds, torch)
    entry("span_attn[B=%d,ctx=%d]" % (B, cur), t, st.attn.algo_bytes(B * cur), nl, "span_attn")
    t = time_kernel_loop([lambda: st.lm_head(xn, ws, out=st.logits)], 10, torch)
    entry("wq_gemm[lm_head bf16 %dx%d]" % (cfg.hidden, cfg.vocab), t, st.lm_head.op.algo_bytes(B), 1, "wq_gemm[lm_head]",
          note="same weights every launch; 1.09 GB >> L2")
    tot = sum(v["us"] * v["launches_per_step"] for v in kern.values())
    for v in kern.values():
        v["share_of_kernel_time"] = round(v["us"] * v["launches_per_step"] / tot, 3)
    return kern


def step_roofline(st, ctx, ms_per_step, hbm_peak):
    wbytes, kvbytes = st.algo_bytes_per_step(ctx)
    sb = wbytes + kvbytes
    return {"algo_bytes": sb, "weights_bytes": wbytes, "kv_bytes": kvbytes,
            "GBps": round(sb / (ms_per_step * 1e-3) / 1e9, 1), "frac": round(sb / (ms_per_step * 1e-3) / 1e9 / hbm_peak, 3),
            "roofline_tok_s": round(st.B / (sb / (hbm_peak * 1e9)), 1)}


DUMP_BYTES = 64_000_000


def dump_outputs(st, out_dir):
    """What the last timed step handed its caller, as DIR/<name>.npy: next_ids (the sampled token ids, float64) and logits
    (float32 [batch, vocab]; under --tp N rank 0's vocabulary shard).  Logits beyond DUMP_BYTES in all are cut to a fixed
    seeded sample of vocabulary columns, whose indices go to logits_columns (float64)."""
    import numpy as np
    ids = st.next_ids.cpu().numpy().astype(np.float64)
    logits = st.logits.float().cpu().numpy()
    out = {"next_ids": ids}
    B, V = logits.shape
    if ids.nbytes + logits.nbytes > DUMP_BYTES:
        n = (DUMP_BYTES - ids.nbytes) // (4 * B + 8)
        cols = np.sort(np.random.default_rng(0).choice(V, n, replace=False))
        out["logits_columns"] = cols.astype(np.float64)
        logits = logits[:, cols]
    out["logits"] = logits
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure_tp(args, world, rank, hbm_peak, torch, dist):
    """Config C4 (BASELINE.json): ONE Qwen2-72B IQ-int4 instance, tensor parallel over all ranks of the job (QKV / gate / up
    column split, o / down row split + all-reduce, vocab-split lm_head), batch 16, ctx 4096, bf16 KV."""
    from b200spark import model
    cfg = model.QWEN2_72B
    B, ctx = args.tp_batch, args.tp_ctx
    K, W = args.steps, 3
    t0 = time.time()
    st = model.DecodeStack(cfg, B, ctx + 3 * K + W + 16, wbits=4, group=-1, kv="none", span=128, tp_rank=rank, tp_size=world,
                           layers=args.tp_layers)
    st.set_context(ctx)
    st.capture()
    build_s = time.time() - t0
    st.ids.copy_(torch.randint(0, cfg.vocab, (B,), generator=torch.Generator().manual_seed(4321), dtype=torch.int64).cuda())
    ms, _ = timed_steps(st, K, W, torch, dist, world)
    ms_step = ms / K
    roof = step_roofline(st, ctx, ms_step, hbm_peak)       # per-rank bytes: the roofline is per GPU
    rec = {"workload": "%s IQ-int4 per-channel, batch %d, ctx %d, bf16 KV, TP=%d (one instance over %d GPUs)" %
                       (cfg.name, B, ctx, world, world),
           "tokens_per_s": round(B * K / (ms * 1e-3), 2), "ms_per_step": round(ms_step, 4), "steps": K, "warmup": W,
           "per_rank_step": roof, "layers": len(st.layers), "build_s": round(build_s, 1),
           "collective": st.collective_probe(K, dist)}
    rec["collective"]["share_of_step"] = round(rec["collective"]["ms_per_step_alone"] / ms_step, 3)
    return rec


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from b200spark import model

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = {"qwen2-7b": model.QWEN2_7B, "llama3-8b": model.LLAMA3_8B, "qwen2-72b": model.QWEN2_72B, "tiny": model.TINY}[args.model]
    B, ctx, K, W = args.batch, args.ctx, args.steps, max(args.warmup, 3)
    tp = args.tp
    if tp > 1 and tp != world:
        raise SystemExit("--tp N must equal the torchrun world size (one rank per GPU)")
    hbm_peak, peak_src = peaks()
    max_len = ctx + W + 3 * K + 16
    t_build = time.time()
    st = model.DecodeStack(cfg, B, max_len, wbits=args.wbits, group=args.group, kv=args.kv, span=args.span,
                           layers=args.layers, tp_rank=rank if tp > 1 else 0, tp_size=tp)
    st.set_context(ctx)
    st.capture()
    t_build = time.time() - t_build

    ids = torch.randint(0, cfg.vocab, (B,), generator=torch.Generator().manual_seed(4321), dtype=torch.int64)
    st.ids.copy_(ids.cuda())
    ms, clocks = timed_steps(st, K, W, torch, dist, world, ClockSampler(local) if rank == 0 else None)
    if args.dump_outputs and rank == 0:
        dump_outputs(st, args.dump_outputs)
    replicas = 1 if tp > 1 else world  # TP: the ranks share one batch; replicas: every rank has its own
    value = replicas * B * K / (ms * 1e-3)
    e2e_s = e2e_steps(st, ids, K, torch, dist, world)
    e2e_val = replicas * B * K / e2e_s
    launches = st.launches_per_step * K
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        traffic = {}

    out = None
    kern = step = None
    if rank == 0:
        kern = kernel_rooflines(st, cfg, hbm_peak, torch, traffic)
        step = step_roofline(st, ctx, ms / K, hbm_peak)

    # ---------------- the metric's other batches on the same weights and caches (every rank takes part: barriers inside)
    batches = {}
    subs = [int(b) for b in args.sub_batches.split(",") if b.strip()] if (tp == 1 and args.sub_batches) else []
    for b in subs:
        if b >= B:
            continue
        st.set_batch(b)
        rewind(st, ctx)
        st.capture()
        st.ids.copy_(ids[:b].cuda())
        ms_b, _ = timed_steps(st, K, W, torch, dist, world)
        rewind(st, ctx)
        e2e_b = e2e_steps(st, ids, K, torch, dist, world)
        rewind(st, ctx)
        rec = {"tokens_per_s": round(replicas * b * K / (ms_b * 1e-3), 2), "ms_per_step": round(ms_b / K, 4), "steps": K, "warmup": W,
               "e2e_tokens_per_s": round(replicas * b * K / e2e_b, 2), "gpu_launches": st.launches_per_step * K}
        if rank == 0:
            rec["step"] = step_roofline(st, ctx, ms_b / K, hbm_peak)
            rec["kernels"] = kernel_rooflines(st, cfg, hbm_peak, torch, traffic)
        batches[str(b)] = rec
    st.set_batch(B)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import decoder_ref as DR
        r = DR.time_cpu_decode(SimpleNamespace(**MODEL_DIMS[args.model]), B, ctx, sample_layers=2, steps=2, warmup=1,
                               threads=physical_cores())
        cpu = {"value": round(r["tokens_per_s"], 3), "unit": "tokens/s", "cores": r["threads"], "kind": "port",
               "sample": "2 of %d decoder layers + lm_head, 2 timed steps after 1 warm-up, bf16 oneDNN matmul via torch CPU, "
                         "fp32 contiguous KV at ctx %d, batch %d; per-layer time x %d layers + head" % (cfg.layers, ctx, B, cfg.layers)}

    # ---------------- config C4 over all ranks (torchrun only)
    tp_rec = None
    if world > 1 and tp == 1 and not args.no_tp_record:
        del st
        torch.cuda.empty_cache()
        tp_rec = measure_tp(args, world, rank, hbm_peak, torch, dist)

    if rank == 0:
        dom = max(kern, key=lambda k: kern[k]["share_of_kernel_time"])
        roof = {"bound": "hbm", "kernel": dom, "achieved": kern[dom]["GBps"], "peak": hbm_peak, "unit": "GB/s",
                "frac": kern[dom]["frac"], "traffic": kern[dom]["traffic"], "peak_source": peak_src,
                "share_of_kernel_time": kern[dom]["share_of_kernel_time"], "step": step}
        if tp > 1:
            roof["step"]["note"] = "per-rank algorithmic bytes; tokens/s is for the whole TP group"
        out = {
            "metric": METRIC, "value": round(value, 2), "unit": "tokens/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(ms / K, 4), "higher_is_better": True, "scaling": "strong" if tp > 1 else "weak", "vs_baseline": None,
            "dtype": "bf16 activations x int%d weights (fp32 accumulate), %s KV" % (args.wbits, args.kv),
            "data": "synthetic (seeded N(0,0.02^2) weights quantized with the IQ formula; N(0,1) KV rows written by the append kernel)",
            "config": {"workload": "%s IQ-int%d%s weight-only decode, batch %d, ctx %d, 1xB200 per replica" %
                                   (cfg.name, args.wbits, "" if args.group == -1 else " g%d" % args.group, B, ctx),
                       "batch": B, "ctx": ctx, "layers": args.layers or cfg.layers, "kv_cache": args.kv, "span": args.span,
                       "parallelism": ("tp%d (column/row split, all-reduce after o_proj and down_proj, vocab-split lm_head)" % tp)
                                      if tp > 1 else "replicas x%d (no data-path collective)" % world,
                       "l2": "inputs larger than L2: %.2f GB streamed per step vs 126 MB L2" % (step["algo_bytes"] / 1e9),
                       "cuda_graph": True, "pdl": os.environ.get("B2_PDL", "1") != "0"},
            "e2e": {"value": round(e2e_val, 2), "unit": "tokens/s", "h2d_bytes_per_step": B * 8, "d2h_bytes_per_step": B * 8},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roof,
            "kernels": kern,
            "batches": batches,
            "cpu_baseline": cpu,
            "build_s": round(t_build, 1),
        }
        if tp_rec is not None:
            out["tp"] = tp_rec
        print(json.dumps(out), flush=True)
    if world > 1:
        # let everybody meet, then leave WITHOUT tearing the communicator down (destroying a process group whose
        # collectives were captured in live CUDA graphs hung on the 2-GPU box); a hard exit after the barrier is clean
        # for torchrun (exit code 0 on every rank)
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)
    return out


def run_reference(args):
    """The reference's CPU path (restated: oracle/decoder_ref.py; the reference CPU binary cannot be built here —
    DESIGN.md §4) on this box's host cores, same config/metric.  Every timed step is a BOUNDED SAMPLE of one decode step:
    2 of the model's decoder layers + final norm + lm_head; `ms_per_step` is what one sampled step really took (so
    steps x ms_per_step is the wall time of the timed region) and `value` scales the per-layer time to the full depth.
    No product code is imported on this path."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import decoder_ref as DR
    dims = MODEL_DIMS[args.model]
    cfg = SimpleNamespace(**dims)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    threads = physical_cores()        # torchrun sets OMP_NUM_THREADS=1: size the pool explicitly
    steps, warmup = max(1, args.steps), max(1, args.warmup)
    r = DR.time_cpu_decode(cfg, args.batch, args.ctx, sample_layers=2, steps=steps, warmup=warmup, threads=threads)
    v = round(r["tokens_per_s"], 3)
    sample = ("each step = 2 of %d decoder layers + final norm + lm_head (value = batch / (per-layer time x %d + head time)), bf16 "
              "oneDNN matmul via torch CPU, fp32 contiguous KV at ctx %d, batch %d, %d timed steps after %d warm-ups" %
              (cfg.layers, cfg.layers, args.ctx, args.batch, steps, warmup))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "tokens/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": round(r["s_per_step_sampled"] * 1e3, 3),
        "ms_per_full_step_extrapolated": round(r["s_per_step_full"] * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16 (dequantized weights, CPU)", "data": "synthetic",
        "config": {"workload": "%s IQ-int%d weight-only decode, batch %d, ctx %d (reference CPU path, dequantized bf16)" %
                               (cfg.name, args.wbits, args.batch, args.ctx), "batch": args.batch, "ctx": args.ctx},
        "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": r["threads"], "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200spark")
    ap.add_argument("--model", default="qwen2-7b")
    ap.add_argument("--batch", type=int, default=int(os.environ.get("B2_BENCH_BATCH", "64")))
    ap.add_argument("--sub-batches", default="8,1", help="other batches of the metric measured on the same weights ('' = none)")
    ap.add_argument("--ctx", type=int, default=2048)
    ap.add_argument("--wbits", type=int, default=4)
    ap.add_argument("--group", type=int, default=-1)
    ap.add_argument("--kv", default="none")
    ap.add_argument("--span", type=int, default=128)
    ap.add_argument("--layers", type=int, default=None, help="debug: fewer layers (INVALID as a bench number)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--tp", type=int, default=1, help="tensor-parallel degree: all ranks of the torchrun job form ONE model instance")
    ap.add_argument("--no-tp-record", action="store_true", help="torchrun: skip the Qwen2-72B TP=N record")
    ap.add_argument("--tp-batch", type=int, default=16)
    ap.add_argument("--tp-ctx", type=int, default=4096)
    ap.add_argument("--tp-layers", type=int, default=None, help="debug: fewer layers in the TP record (INVALID as a bench number)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the next_ids / logits of the last timed step as DIR/<name>.npy (float32 / float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the b200spark arm's outputs")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
