"""ctypes binding of libspb200.so (the C ABI declared in include/spb200.h).

There is no CPU fallback: importing works anywhere, but touching `lib()` without the built
library, or calling a kernel without a CUDA device, raises.  Build with
`python -c "import __graft_entry__ as g; g.build()"` (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from ctypes import c_char_p, c_float, c_int, c_int64, c_longlong, c_uint64, c_void_p
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libspb200.so")
SOURCES = ["api.cu", "collate.cu", "decode_stack.cu", "gemm.cu", "ffn.cu", "ffn_bwd.cu", "rowops.cu", "embed_scatter.cu", "attention.cu", "attention_tc.cu", "attention_bwd_tc.cu", "latents.cu", "heads.cu", "head_ce.cu", "tables.cu", "optim.cu"]

_P, _I, _F, _L, _U64 = c_void_p, c_int, c_float, c_int64, c_uint64
_U32 = ctypes.c_uint32

# name -> argument ctypes (all functions return int); mirrors include/spb200.h line by line
SIGNATURES = {
    "spb_cast_f32_bf16": [_P, _P, _L, _P, _I, _P],
    "spb_colsum": [_P, _I, _I, _P, _I, _I, _P],
    "spb_gemm_bf16": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _I, _P, _I, _I, _I, _P, _P],
    "spb_layer_norm_fwd": [_P, _I, _I, _P, _P, _P, _I, _P, _I, _I, _P, _P, _I, _I, _F, _P],
    "spb_layer_norm_bwd": [_P, _I, _P, _I, _I, _P, _P, _P, _P, _I, _P, _I, _P, _I, _I, _P, _P, _P, _I, _P, _I, _P, _I, _I, _P],
    "spb_glu_fwd": [_P, _P, _I, _I, _F, _U64, _P, _P],
    "spb_sample_fields": [_P, _I, _P, _P, _P, _P, _P, _I, _I, _F, _U64, _P, _P, _I, _I, _I, _P, _P],
    "spb_sample_fields_filtered": [_P, _I, _P, _P, _P, _P, _P, _I, _I, _F, _U64, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P],
    "spb_decode_stack_step": [_P, _P, _I, _P, _P, _P, _I, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _F, _P, _I, _P, _I, _P],
    "spb_gather_at_pos": [_P, _P, _P, _P, _I, _P, _I, _I, _P],
    "spb_session_begin": [_P, _I, _P, _P, _P, c_longlong, _P],
    "spb_unpack_batch": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _U32, _U32, _I, c_longlong, _I, _P],
    "spb_ffn_fwd": [_P, _I, _P, _P, _P, _P, _I, _P, _I, _P, _P, _I, _I, _I, _F, _U64, _P, _P],
    "spb_ffn_bwd": [_P, _I, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _U64, _P, _P],
    "spb_multi_copy": [_P, _P, _P, _I, _P],
    "spb_multi_add_f32": [_P, _P, _P, _I, _P],
    "spb_transpose_bf16": [_P, _I, _P, _I, _I, _P],
    "spb_glu_bwd": [_P, _P, _P, _P, _I, _I, _F, _U64, _P, _P],
    "spb_table_build_fwd": [_P, _I, _P, _P, _P],
    "spb_table_build_bwd": [_P, _I, _P, _P, _P],
    "spb_embed_ln_fwd": [_P, _I, _P, _P, _I, _P, _P, _P, _I, _P, _P, _I, _F, _P],
    "spb_embed_ln_bwd": [_P, _I, _P, _I, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P],
    "spb_attention_fwd": [_P, _I, _P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _F, _U64, _P, _P],
    "spb_attention_fwd_tc": [_P, _I, _P, _P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _I, _F, _U64, _P, _P],
    "spb_attention_bwd_tc": [_P, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _F, _U64, _P, _P],
    "spb_attention_bwd": [_P, _I, _P, _P, _P, _P, _I, _P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _F, _U64, _P, _I, _P],
    "spb_attention_decode": [_P, _I, _P, _I, c_longlong, _P, _I, _P, _P, _I, _I, _I, _I, _I, _I, _P, _I, _P],
    "spb_latent_level_fwd": [_P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "spb_latent_level_bwd": [_P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "spb_mmd_fwd_bwd": [_P, _P, _P, _I, _I, _I, _P, _P, _P, _P],
    "spb_head_ce": [_P, _I, _P, _I, _I, _P, _I, c_longlong, _P, _P, _P, _I, _P, _P, _P, _I, _P],
    "spb_adamw_step": [_P, _P, _P, _P, _P, _L, _P, _F, _F, _F, _F, _F, _F, _F, _P, _P, _P],
    "spb_gemm_bf16_rowdot": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _I, _P, _I, _I, _P],
    "spb_ce_rows": [_P, _I, _P, _I, _I, c_longlong, _P, _P, _P, _I, _P, _I, _P],
    "spb_clf_heads": [_P, _I, _P, _P, _I, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _I, _I, _F, _U64, _P, _I, _P],
    "spb_clf_logits": [_P, _I, _P, _P, _P, _I, _I, _I, _P],
}

_lib: Optional[ctypes.CDLL] = None


NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--use_fast_math", "-Xcompiler", "-fPIC"]
BUILD_DIR = os.path.join(os.path.dirname(_HERE), "build")


def _digest(paths) -> str:
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for p in paths:
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every kernel for sm_100a into scoreperformer_b200/csrc/libspb200.so (in-tree, git-ignored).

    One nvcc process per .cu (in parallel), objects cached under build/ by the hash of the source + common.cuh + flags, so
    only edited files recompile; the library is relinked whenever an object changed.  A shipped prebuilt library is kept
    only if it was linked from exactly the current sources (the hash list is stored next to it)."""
    from concurrent.futures import ThreadPoolExecutor
    common = os.path.join(CSRC, "common.cuh")
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    digests = [_digest([s, common]) for s in srcs]
    stamp = LIB_PATH + ".srchash"
    want = "\n".join(digests)
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp) and open(stamp).read() == want:
        return LIB_PATH
    import shutil
    if shutil.which("nvcc") is None:
        if os.path.exists(LIB_PATH):      # GPU box without a toolchain: the snapshot's library is what there is
            return LIB_PATH
        raise RuntimeError("nvcc not found and no prebuilt libspb200.so: scoreperformer_b200 has no CPU / PyTorch fallback")
    os.makedirs(BUILD_DIR, exist_ok=True)
    objs = [os.path.join(BUILD_DIR, f"{os.path.splitext(os.path.basename(s))[0]}.{d}.o") for s, d in zip(srcs, digests)]

    def compile_one(job):
        src, obj = job
        if os.path.exists(obj) and not force:
            return None
        cmd = ["nvcc"] + NVCC_FLAGS + ["-c", "-o", obj, src]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or res.returncode != 0:
            print(" ".join(cmd))
            print(res.stdout + res.stderr)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed on {os.path.basename(src)}:\n" + res.stderr[-4000:])
        return obj

    with ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 4)) as pool:
        list(pool.map(compile_one, zip(srcs, objs)))
    cmd = ["nvcc", "-shared", "-o", LIB_PATH] + objs
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("linking libspb200.so failed:\n" + res.stderr[-4000:])
    with open(stamp, "w") as f:
        f.write(want)
    # drop objects of older source versions
    keep = set(objs)
    for name in os.listdir(BUILD_DIR):
        path = os.path.join(BUILD_DIR, name)
        if name.endswith(".o") and path not in keep:
            os.remove(path)
    return LIB_PATH


def lib() -> ctypes.CDLL:
    """The loaded library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: scoreperformer_b200 has no CPU / PyTorch fallback. "
                "Run `python -c \"import __graft_entry__ as g; g.build()\"` (needs nvcc).")
        handle = ctypes.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.argtypes = argtypes
            fn.restype = c_int
        handle.spb_last_error.restype = c_char_p
        handle.spb_last_error.argtypes = []
        handle.spb_abi_version.restype = c_int
        _lib = handle
    return _lib


def check(rc: int, name: str) -> None:
    if rc != 0:
        msg = lib().spb_last_error().decode(errors="replace")
        raise RuntimeError(f"{name} failed (code {rc}): {msg}")
