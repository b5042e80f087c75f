"""ctypes binding of the C-ABI kernel library (include/dahitra_b200.h) and its in-tree build.

The shared object lives next to this file (``dahitra_b200/libdahitra_b200.so``) so it travels with the
source tree; it is produced by ``build()`` (``nvcc -gencode arch=compute_100a,code=sm_100a``).
There is no fallback: if the library is missing or fails to load, every native entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libdahitra_b200.so")
SOURCES = ["conv_ffma.cu", "conv_tc.cu", "conv_tc2.cu", "conv_tc3.cu", "split.cu", "tokens.cu", "decoder.cu", "decoder_tc.cu", "stem_tc.cu", "classifier.cu", "train_decoder.cu", "train_tokens.cu", "prepare.cu", "aux.cu", "forward.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]

_lock = threading.Lock()
_lib = None


def _sources():
    return [os.path.join(_CSRC, s) for s in SOURCES if os.path.exists(os.path.join(_CSRC, s))]


STAMP_PATH = LIB_PATH + ".stamp"


def _deps():
    deps = _sources() + [os.path.join(_HERE, "..", "include", "dahitra_b200.h")]
    deps += [os.path.join(_CSRC, f) for f in sorted(os.listdir(_CSRC)) if f.endswith(".cuh")]
    return [d for d in deps if os.path.exists(d)]


def _source_hash() -> str:
    """content hash of everything the library is compiled from (sources, headers, flags)"""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS + [os.environ.get("DAHITRA_DEBUG_BUILD", "0")]).encode())
    for d in _deps():
        h.update(os.path.basename(d).encode() + b"\0")
        with open(d, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def needs_build() -> bool:
    """True when the in-tree library is missing or was built from other sources.  The build leaves a content hash of its inputs
    next to the library (git-ignored like the library, travels with the tree): file times do not survive every copy of a tree.
    Without a stamp (a library built before stamps existed) the file times decide, and a library they call fresh is stamped."""
    if not os.path.exists(LIB_PATH):
        return True
    if os.path.exists(STAMP_PATH):
        with open(STAMP_PATH) as f:
            return f.read().strip() != _source_hash()
    t = os.path.getmtime(LIB_PATH)
    if any(os.path.getmtime(d) > t for d in _deps()):
        return True
    _write_stamp()
    return False


def _write_stamp():
    try:
        with open(STAMP_PATH + ".tmp", "w") as f:
            f.write(_source_hash() + "\n")
        os.replace(STAMP_PATH + ".tmp", STAMP_PATH)
    except OSError:
        pass                                    # read-only tree: the file times keep deciding


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ for sm_100a (objects in parallel, then one link) into the in-tree shared object;
    cross-compiles without a GPU."""
    if not force and not needs_build():
        return LIB_PATH
    import tempfile
    from concurrent.futures import ThreadPoolExecutor
    nvcc = os.environ.get("NVCC", "nvcc")
    cflags = [f for f in NVCC_FLAGS if f != "-shared"]
    if os.environ.get("DAHITRA_DEBUG_BUILD") == "1":      # bounded mbarrier waits that trap + printf instead of hanging
        cflags.append("-DDH_MBAR_TIMEOUT")
    with tempfile.TemporaryDirectory(prefix="_build_", dir=_HERE) as tmp:            # in-tree scratch (objects are git-ignored)
        def compile_one(src):
            obj = os.path.join(tmp, os.path.basename(src) + ".o")
            cmd = [nvcc] + cflags + ["-c", src, "-o", obj]
            if verbose:
                print(" ".join(cmd), flush=True)
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed on %s:\n%s%s" % (src, r.stdout, r.stderr))
            return obj
        with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
            objs = list(ex.map(compile_one, _sources()))
        cmd = [nvcc] + NVCC_FLAGS + objs + ["-o", LIB_PATH + ".tmp"]
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc link failed:\n" + r.stdout + r.stderr)
    os.replace(LIB_PATH + ".tmp", LIB_PATH)
    _write_stamp()
    return LIB_PATH


EXAMPLE_SRC = os.path.join(_HERE, "..", "examples", "dahitra_infer.c")
EXAMPLE_BIN = os.path.join(_HERE, "..", "examples", "bin", "dahitra_infer")


def build_example(force: bool = False, verbose: bool = False) -> str:
    """Compile the plain-C host of the C ABI (examples/dahitra_infer.c: C99, gcc, the CUDA runtime linked statically) against the
    in-tree library.  No Python or PyTorch is involved in what it runs; the binary is git-ignored and travels with the tree."""
    src, out = os.path.abspath(EXAMPLE_SRC), os.path.abspath(EXAMPLE_BIN)
    deps = [src, LIB_PATH, os.path.join(_HERE, "..", "include", "dahitra_b200.h")]
    if not force and os.path.exists(out) and all(os.path.getmtime(d) <= os.path.getmtime(out) for d in deps):
        return out
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    cmd = [os.environ.get("CC", "gcc"), "-std=c99", "-O2", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(_HERE, "..", "include"),
           "-I", os.path.join(cuda, "include"), src, "-L", _HERE, "-ldahitra_b200", "-L", os.path.join(cuda, "lib64"),
           "-l:libcudart_static.a", "-ldl", "-lpthread", "-lrt", "-Wl,-rpath,$ORIGIN/../../dahitra_b200", "-o", out + ".tmp"]
    if verbose:
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("building examples/dahitra_infer.c failed:\n" + r.stdout + r.stderr)
    os.replace(out + ".tmp", out)
    return out


# (name, restype, argtypes) — must match include/dahitra_b200.h exactly
_P, _I, _LL, _SZ = C.c_void_p, C.c_int, C.c_longlong, C.c_size_t
SIGNATURES = {
    "dahitra_version": (_I, []),
    "dahitra_error_string": (C.c_char_p, [_I]),
    "dahitra_weight_slot_name": (C.c_char_p, [_I]),
    "dahitra_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I, _I]),
    "dahitra_prepare_weights": (_LL, [_P, _I, _I, _I, _P, _LL, _P]),
    "dahitra_forward": (_I, [_P, _I, _P, _P, _LL, _P, _P, _P, _SZ, _I, _I, _I, _I, _I, _I, _P]),
    "dahitra_forward_profiled": (_I, [_P, _I, _P, _P, _LL, _P, _P, _P, _SZ, _I, _I, _I, _I, _I, _I, _P,
                                      _I, _P, _P, _P, _P]),
    "dahitra_conv2d": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _I, _P, _I, _P]),
    "dahitra_conv2d_up2_tc": (_I, [_P, _I, _I, _I, _P, _P, _I, _P, _I, _P]),
    "dahitra_stem": (_I, [_P, _LL, _I, _I, _I, _P, _P, _P, _P]),
    "dahitra_stem_tc": (_I, [_P, _LL, _I, _I, _I, _P, _P, _P, _I, _P]),
    "dahitra_maxpool3x3s2": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "dahitra_squeeze_tokens": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _P]),
    "dahitra_token_encoder": (_I, [_P, _I, _I, _P, _I, _I, _P, _P]),
    "dahitra_decoder_tables": (_I, [_P, _I, _I, _I, _P, _I, _I, _P, _P]),
    "dahitra_pixel_decoder": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _I, _P, _P]),
    "dahitra_decoder_tables_tc": (_I, [_P, _I, _I, _I, _P, _I, _I, _P, _P]),
    "dahitra_pixel_decoder_tc": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _I, _I, _P, _P]),
    "dahitra_confusion_matrix": (_I, [_P, _P, _LL, _I, _P, _P]),
    "dahitra_prepare_input_u8": (_I, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "dahitra_classifier": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "dahitra_split_pack": (_I, [_P, _LL, _P, _P]),
    "dahitra_split_unpack": (_I, [_P, _LL, _P, _P]),
    "dahitra_maxpool3x3s2_split": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "dahitra_pixel_decoder_train_blocks": (_I, [_I]),
    "dahitra_pixel_decoder_train_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "dahitra_pixel_decoder_train_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "dahitra_tokenizer_train_chunks": (_I, [_I]),
    "dahitra_tokenizer_train_fwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "dahitra_tokenizer_train_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "dahitra_pixel_decoder_train_fwd_ex": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "dahitra_pixel_decoder_train_bwd_ex": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "dahitra_tokenizer_train_fwd_ex": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "dahitra_tokenizer_train_bwd_ex": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "dahitra_conv2d_split": (_I, [_P, _P, _I, _I, _LL, _LL, _I, _I, _I, _I, _I, _I, _P, _P, _P, _I, _I, _P, _I, _I, _P, _P, _P]),
    "dahitra_maxpool3x3s2_h16": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "dahitra_classifier_h16": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
}


class DhTensor(C.Structure):
    """struct dh_tensor of include/dahitra_b200.h"""
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("dtype", C.c_int), ("ndim", C.c_int), ("shape", C.c_longlong * 4)]


def load():
    """Return the loaded library (ctypes.CDLL) or raise — never returns a stub."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"dahitra_b200: {LIB_PATH} is missing — run `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(nvcc, sm_100a). There is no fallback path.")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)          # AttributeError if the .so does not export it
                fn.restype, fn.argtypes = res, args
            _lib = lib
        return _lib


def check(rc: int, what: str = "dahitra"):
    if rc != 0:
        msg = load().dahitra_error_string(rc)
        raise RuntimeError(f"{what} failed with code {rc}: {msg.decode() if msg else '?'}")
