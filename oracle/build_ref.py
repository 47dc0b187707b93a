"""Build oracle/_ref/libdashinfer_ref.so — the UNMODIFIED reference GPU code for the KV-cache half of the hot path,
compiled from the sources where they lie under /root/reference (nothing is copied into the repo).

TEST INFRASTRUCTURE: only tests/ and __graft_entry__.build() use this.  The output is git-ignored;
tests/golden/make_ref_pin.py runs it on a GPU to record the reference's own results, to which tests/test_ref_pin_gpu.py
pins oracle/kvcache_ref.py and the b200spark kernels.

What is compiled (nvcc directly, no cmake; -DNDEBUG like the reference's Release build):
  * span-attention/src/**/*.cu|*.cpp          the span-attention library (span::CreateHandle/Run ...), header-only
                                              CUTLASS from span-attention/thirdparty/cutlass/include
  * csrc/core/kernel/cuda/cache/decoder_cache_append_{bf16,fp16}.cu, context_span_copy_{bf16,fp16}.cu
                                              with three stub headers from oracle/ref_stubs/ standing in for engine
                                              headers that need glog/protobuf/cublas (no kernel code in the stubs)
  * oracle/ref_shim.cu                        extern "C" entry points for ctypes
Target: sm_100 (plain, the reference has no Blackwell-specific code; its mma.sync kernels run as they are).

The CPU x86 path of the reference cannot be built at all (oneDNN/MKL tarballs are git-LFS stubs) — DESIGN.md §4.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("B2_REFERENCE", "/root/reference")
OUT = os.path.join(HERE, "_ref")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
SO = os.path.join(OUT, "libdashinfer_ref.so")


def sources():
    sa = os.path.join(REF, "span-attention", "src")
    srcs = []
    for root, _, files in os.walk(sa):
        for f in sorted(files):
            if f.endswith((".cu", ".cpp")):
                srcs.append(os.path.join(root, f))
    cache = os.path.join(REF, "csrc", "core", "kernel", "cuda", "cache")
    for f in ("decoder_cache_append_bf16.cu", "decoder_cache_append_fp16.cu", "context_span_copy_bf16.cu",
              "context_span_copy_fp16.cu"):
        srcs.append(os.path.join(cache, f))
    srcs.append(os.path.join(HERE, "ref_shim.cu"))
    return sorted(srcs)


def build(force=False, verbose=False):
    if not os.path.isdir(REF):
        return SO if os.path.exists(SO) else None   # GPU box: use the prebuilt file
    srcs = sources()
    if not force and os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(s) for s in srcs + [__file__]):
        return SO
    os.makedirs(OUT, exist_ok=True)
    sa = os.path.join(REF, "span-attention")
    inc = ["-I", os.path.join(HERE, "ref_stubs"),                       # stubs first: shadow the engine headers
           "-I", os.path.join(sa, "include", "spanattn"), "-I", os.path.join(sa, "include"), "-I", os.path.join(sa, "src"),
           "-I", os.path.join(sa, "thirdparty", "cutlass", "include"),
           "-I", os.path.join(REF, "csrc", "common"), "-I", os.path.join(REF, "csrc", "core", "kernel"),
           "-I", os.path.join(REF, "csrc", "device"), "-I", os.path.join(REF, "csrc")]        # <cuda/cudabfloat16_impl.hpp>
    flags = ["-gencode", "arch=compute_100,code=sm_100", "-std=c++17", "-O2", "-DNDEBUG", "-DENABLE_BF16", "-DENABLE_FP16",
             "-DENABLE_CUDA", "--expt-relaxed-constexpr", "--extended-lambda", "--use_fast_math", "-Xcompiler", "-fPIC",
             "-x", "cu", "-w"]

    def one(src):
        obj = os.path.join(OUT, os.path.relpath(src, "/").replace("/", "_") + ".o")
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= os.path.getmtime(src):
            return obj
        cmd = [NVCC] + flags + inc + ["-c", src, "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            sys.stdout.write(r.stdout)
            raise RuntimeError("reference build failed: " + src)
        return obj

    with ThreadPoolExecutor(max_workers=int(os.environ.get("B2_REF_JOBS", "8"))) as ex:
        objs = list(ex.map(one, srcs))
    r = subprocess.run([NVCC, "-gencode", "arch=compute_100,code=sm_100", "-shared", "-o", SO] + objs,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stdout.write(r.stdout)
        raise RuntimeError("reference link failed")
    return SO


if __name__ == "__main__":
    print("built:", build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
