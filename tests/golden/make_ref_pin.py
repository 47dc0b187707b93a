"""Reference results for tests/test_ref_pin_gpu.py, computed by the REFERENCE's own GPU code on the seeded inputs the
tests draw: oracle/_ref/libdashinfer_ref.so, the unmodified span-attention library and span-cache writers of
modelscope/dash-infer, built by oracle/build_ref.py (B2_REFERENCE=<dash-infer checkout>).  Needs a GPU:
    python tests/golden/make_ref_pin.py [OUT_DIR]         (default: tests/golden)
Writes ref_pin.json (SHA-256 of the span bytes DecoderCacheAppendLauncher / ContextSpanCopyLauncher wrote and of the Q rows
the append gathered) and ref_pin_attn.npz (span::Run outputs as bf16 bit patterns, uint16 [batch, heads * 128])."""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.join(ROOT, "dash-infer_b200", "python"), ROOT, os.path.dirname(HERE)):
    sys.path.insert(0, p)
import test_ref_pin_gpu as T  # noqa: E402
from b200spark import ops  # noqa: E402
from oracle import ref_lib as RL  # noqa: E402


def main(out_dir):
    lib = RL.load()
    assert lib is not None, "oracle/_ref/libdashinfer_ref.so is not built (python oracle/build_ref.py)"
    print(lib.ref_version().decode())

    def ref_append(cache, qkv, pos):
        c = cache.cfg
        q = torch.empty(qkv.shape[0], c.n_heads * c.head_size, dtype=qkv.dtype, device=qkv.device)
        return RL.cache_append(lib, cache.k_tab, cache.v_tab, q, qkv, pos, c.n_heads, c.n_groups, c.span_len,
                               c.max_spans_per_seq, c.quant_mode)

    res = {"reference": lib.ref_version().decode(), "append": {}, "attention": {}, "context_copy": {}}
    outs = {}
    for mode in T.MODES:
        for span in T.APPEND_SPANS:
            cache, q, _ = T.append_fill(ref_append, mode, span)
            res["append"]["mode%d_span%d" % (mode, span)] = T.digest(cache, q)
    for mode in T.MODES:
        for case, (lens, nH, nG, span) in enumerate(T.CASES):
            key = "mode%d_case%d" % (mode, case)
            cache, q_last = T.attention_fill(ref_append, mode, case)
            res["attention"][key] = T.digest(cache, q_last)
            out = torch.empty_like(q_last)
            RL.span_attn(lib, out, q_last, cache.k_tab, cache.v_tab, lens, nH, nG, span, cache.max_spans, mode, T.ATTN_SCALE)
            torch.cuda.synchronize()
            outs[key] = out.cpu().view(torch.int16).numpy().view(np.uint16)
    for mode in T.MODES:
        for span, seq in T.CONTEXT_SHAPES:
            cache = ops.SpanCache(1, seq, 8, 2, span, mode)
            RL.context_span_copy(lib, cache.k_tab[0], T.context_src(mode, span, seq), 2, span, seq, mode)
            torch.cuda.synchronize()
            res["context_copy"]["mode%d_span%d_seq%d" % (mode, span, seq)] = T.digest(cache)
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "ref_pin.json"), "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(os.path.join(out_dir, "ref_pin_attn.npz"), **outs)
    print("wrote", out_dir)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)
