"""ctypes binding of libstcd_b200.so (include/stcd_b200.h) and its in-tree nvcc build.

The library is built IN-TREE (``stcd_b200/libstcd_b200.so``) so it travels to the GPU box with the
repo snapshot.  There is no CPU fallback: if the library is missing, or no sm_100 device is
visible, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
REPO_DIR = PKG_DIR.parent
LIB_PATH = PKG_DIR / "libstcd_b200.so"
CSRC = PKG_DIR / "csrc"
HEADER = REPO_DIR / "include" / "stcd_b200.h"

MAX_SRC = 6
MAX_PHASE = 4

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
]


class StcdError(RuntimeError):
    pass


def _sources():
    return sorted(CSRC.glob("*.cu")) + sorted(CSRC.glob("*.cuh")) + [HEADER]


STAMP_PATH = PKG_DIR / "libstcd_b200.so.srchash"      # sha256 of the sources the .so was built from (travels with it)
LOCK_PATH = PKG_DIR / ".build.lock"


def _source_hash() -> str:
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for src in _sources():
        h.update(src.name.encode())
        h.update(src.read_bytes())
    return h.hexdigest()


def needs_build() -> bool:
    """Stale when the .so is missing or was built from other sources (content hash, not mtimes: a snapshot copied
    to a GPU box does not keep them)."""
    if not LIB_PATH.exists():
        return True
    try:
        return STAMP_PATH.read_text().strip() != _source_hash()
    except OSError:
        t = LIB_PATH.stat().st_mtime          # no stamp (built by hand): fall back to mtimes
        return any(s.stat().st_mtime > t for s in _sources())


def build(force: bool = False, verbose: bool = False) -> Path:
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> stcd_b200/libstcd_b200.so

    Safe under torchrun: ranks serialise on a file lock, the compiler writes a temporary file that is renamed
    over the library (no rank can dlopen a half-written .so) and whoever gets the lock second finds it fresh."""
    import fcntl
    import tempfile
    with open(LOCK_PATH, "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():
                return LIB_PATH
            nvcc = os.environ.get("NVCC", "nvcc")
            fd, tmp = tempfile.mkstemp(prefix=".libstcd_b200.", suffix=".so.tmp", dir=str(PKG_DIR))
            os.close(fd)
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["--threads", "0", "-o", tmp] + [str(f) for f in sorted(CSRC.glob("*.cu"))]
            try:
                r = subprocess.run(cmd, capture_output=True, text=True)
                if r.returncode != 0:
                    raise StcdError(f"nvcc failed ({' '.join(cmd)}):\n{r.stdout}\n{r.stderr}")
                os.chmod(tmp, 0o755)
                os.replace(tmp, LIB_PATH)
                STAMP_PATH.write_text(_source_hash() + "\n")
            finally:
                if os.path.exists(tmp):
                    os.unlink(tmp)
            if verbose:
                print(r.stderr)
            return LIB_PATH
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


class Chunk(C.Structure):
    _fields_ = [("src", C.c_int16), ("c0", C.c_int16), ("by", C.c_int16), ("bx", C.c_int16),
                ("n_off", C.c_int32), ("tap_begin", C.c_int16), ("n_taps", C.c_int16)]


class Tap(C.Structure):
    _fields_ = [("ty", C.c_int16), ("tx", C.c_int16)]


class Phase(C.Structure):
    _fields_ = [("chunk_begin", C.c_int32), ("chunk_count", C.c_int32), ("oy", C.c_int32), ("ox", C.c_int32),
                ("w_block", C.c_int32), ("n_blocks", C.c_int32)]


class ConvDesc(C.Structure):
    _fields_ = [
        ("n_src", C.c_int32),
        ("src", C.c_int32 * MAX_SRC),
        ("src_sy", C.c_int32 * MAX_SRC),
        ("src_sx", C.c_int32 * MAX_SRC),
        ("src_ey", C.c_int32 * MAX_SRC),
        ("src_ex", C.c_int32 * MAX_SRC),
        ("hg", C.c_int32), ("wg", C.c_int32),
        ("img_mult", C.c_int32),
        ("pair", C.c_int32),
        ("weights", C.POINTER(C.c_uint16)),
        ("w_elems", C.c_int64),
        ("kc", C.c_int32),
        ("n_tile", C.c_int32),
        ("cout", C.c_int32),
        ("cout_pad", C.c_int32),
        ("n_phase", C.c_int32),
        ("phase", Phase * MAX_PHASE),
        ("chunks", C.POINTER(Chunk)),
        ("n_chunks", C.c_int32),
        ("taps", C.POINTER(Tap)),
        ("n_taps", C.c_int32),
        ("osy", C.c_int32), ("osx", C.c_int32),
        ("scale", C.POINTER(C.c_float)),
        ("shift", C.POINTER(C.c_float)),
        ("scale2", C.POINTER(C.c_float)),
        ("shift2", C.POINTER(C.c_float)),
        ("relu", C.c_int32),
        ("res", C.c_int32),
        ("out0", C.c_int32), ("out0_coff", C.c_int32),
        ("out_raw", C.c_int32),
        ("out_pool", C.c_int32),
        ("out_diff", C.c_int32),
        ("out_ext", C.c_int32),
        ("out0_s2d", C.c_int32),
        ("fold_cs", C.c_int32), ("fold_cout", C.c_int32),
        ("act_pre", C.c_int32), ("act_alpha", C.c_float),
        ("xf_cs", C.c_int32),
    ]


class SegHeadDesc(C.Structure):
    _fields_ = [("src", C.c_int32), ("c", C.c_int32), ("weight", C.POINTER(C.c_float)), ("bias", C.c_float),
                ("out_ext", C.c_int32), ("diff_src", C.c_int32)]


class BitDesc(C.Structure):
    _fields_ = [("c", C.c_int32), ("token_len", C.c_int32), ("heads", C.c_int32), ("mlp", C.c_int32),
                ("n_enc", C.c_int32), ("n_dec", C.c_int32), ("inner_enc", C.c_int32), ("inner_dec", C.c_int32),
                ("softmax", C.c_int32),
                ("conv_a", C.POINTER(C.c_float)), ("pos", C.POINTER(C.c_float)), ("enc", C.POINTER(C.c_float)),
                ("dec", C.POINTER(C.c_float))]


class EcamDesc(C.Structure):
    _fields_ = [
        ("src", C.c_int32 * 4),
        ("c", C.c_int32), ("n_class", C.c_int32), ("r", C.c_int32), ("r1", C.c_int32),
        ("ca_fc1", C.POINTER(C.c_float)), ("ca_fc2", C.POINTER(C.c_float)),
        ("ca1_fc1", C.POINTER(C.c_float)), ("ca1_fc2", C.POINTER(C.c_float)),
        ("w_final", C.POINTER(C.c_float)), ("b_final", C.POINTER(C.c_float)),
        ("out_ext", C.c_int32),
    ]


ABI_VERSION = 21
PRECISION_BF16, PRECISION_SPLIT = 0, 1        # enum stcd_precision

# every symbol include/stcd_b200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("stcd_last_error", C.c_char_p, []),
    ("stcd_abi_version", C.c_int, []),
    ("stcd_device_count", C.c_int, []),
    ("stcd_plan_create", C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    ("stcd_plan_destroy", None, [C.c_void_p]),
    ("stcd_plan_add_tensor", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    ("stcd_plan_add_conv", C.c_int, [C.c_void_p, C.POINTER(ConvDesc)]),
    ("stcd_plan_add_input_pack", C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    ("stcd_plan_add_input_pack_s2d", C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    ("stcd_plan_add_input_pack_u8", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    ("stcd_plan_add_maxpool_s2d", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    ("stcd_plan_add_seg_head", C.c_int, [C.c_void_p, C.c_void_p]),
    ("stcd_plan_add_absdiff", C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    ("stcd_plan_add_subdiff", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    ("stcd_plan_add_channel_gate", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float),
                                             C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int]),
    ("stcd_plan_add_bit_transformer", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    ("stcd_plan_add_channel_attention", C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int, C.c_int,
                                                  C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    ("stcd_plan_add_spatial_gate", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                             C.POINTER(C.c_float)]),
    ("stcd_plan_add_global_local_gate", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    ("stcd_plan_add_csam_gate", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    ("stcd_plan_add_vffm", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    ("stcd_plan_add_sum", C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.c_int, C.c_int]),
    ("stcd_plan_add_graph_conv", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    ("stcd_plan_add_layernorm", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                          C.c_float]),
    ("stcd_plan_add_sr_attention", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float]),
    ("stcd_plan_add_dwconv3x3", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int]),
    ("stcd_plan_add_bilinear_up", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    ("stcd_plan_add_ecam_head", C.c_int, [C.c_void_p, C.c_void_p]),
    ("stcd_plan_finalize", C.c_int, [C.c_void_p]),
    ("stcd_plan_tensor_copy", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_int]),
    ("stcd_plan_read_trace", C.c_int64, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    ("stcd_plan_workspace_bytes", C.c_int64, [C.c_void_p]),
    ("stcd_plan_launches", C.c_int64, [C.c_void_p, C.c_int]),
    ("stcd_forward", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_void_p]),
    ("stcd_forward_u8", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_void_p]),
    ("stcd_forward_host_u8", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int]),
    ("stcd_forward_profile", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_void_p,
                                       C.POINTER(C.c_float), C.c_int]),
    ("stcd_forward_host", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int]),
    ("stcd_confusion_add_batch", C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_int64, C.c_int64,
                                           C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("stcd_binarise_mask", C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    ("stcd_knn_graph", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    ("stcd_max_relative", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_void_p, C.c_void_p]),
]

_lib = None


def lib() -> C.CDLL:
    """Load libstcd_b200.so (building it if nvcc is available and it is stale/missing)."""
    global _lib
    if _lib is not None:
        return _lib
    override = os.environ.get("STCD_LIB")      # development: A/B a previously built library (tools/r2_ab.sh); never set in tests / bench
    if override:
        handle = C.CDLL(override)
    elif needs_build():
        try:
            build()
        except (StcdError, FileNotFoundError) as e:
            if not LIB_PATH.exists():
                raise StcdError(f"libstcd_b200.so is missing and could not be built: {e}") from e
            if os.environ.get("STCD_ALLOW_STALE", "0") != "1":
                # never serve kernels older than the sources silently (ABI_VERSION only catches struct changes)
                raise StcdError("libstcd_b200.so is older than stcd_b200/csrc and the rebuild failed "
                                f"(set STCD_ALLOW_STALE=1 to load it anyway): {e}") from e
            import warnings
            warnings.warn(f"loading a STALE libstcd_b200.so (rebuild failed: {e})", RuntimeWarning)
    if not override:
        handle = C.CDLL(str(LIB_PATH))
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(handle, name)
        fn.restype = restype
        fn.argtypes = argtypes
    if handle.stcd_abi_version() != ABI_VERSION:
        raise StcdError("libstcd_b200.so ABI version mismatch")
    _lib = handle
    return handle


def check(code: int, what: str = "") -> int:
    if code != 0:
        msg = lib().stcd_last_error().decode("utf-8", "replace")
        raise StcdError(f"{what}: {msg} (code {code})" if what else f"{msg} (code {code})")
    return code


def check_id(value: int, what: str = "") -> int:
    if value < 0:
        msg = lib().stcd_last_error().decode("utf-8", "replace")
        raise StcdError(f"{what}: {msg} (code {-value})")
    return value
