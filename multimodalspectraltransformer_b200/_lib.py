"""ctypes binding of libmmt_b200.so (C ABI declared in include/mmt_b200.h).

The library is built in-tree with nvcc for sm_100a (``build()``); there is no
CPU fallback: if the shared object is missing or fails to load, every entry point
of the package raises.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_HERE, "libmmt_b200.so")
SOURCES = [os.path.join(_HERE, "csrc", "engine.cu")]
HEADER = os.path.join(ROOT, "include", "mmt_b200.h")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]

# every symbol include/mmt_b200.h declares (tests check the .so exports all of them)
EXPORTS = [
    "mmt_abi_version", "mmt_last_error", "mmt_weight_count", "mmt_weight_name", "mmt_weight_numel",
    "mmt_weight_offset", "mmt_weight_total", "mmt_create", "mmt_destroy", "mmt_memory_len",
    "mmt_mask_is_float", "mmt_encode", "mmt_spectra_equal", "mmt_decode", "mmt_decode_memory_streams", "mmt_decode_until_eos", "mmt_decode_controlled", "mmt_teacher_forced", "mmt_teacher_forced_scores", "mmt_beam_search", "mmt_sample_without_replacement", "mmt_sbs_select_step", "mmt_philox_increment",
    "mmt_pack_tokens_u8", "mmt_unpack_tokens_u8", "mmt_pack_tokens_u8_seqmajor", "mmt_unpack_tokens_u8_seqmajor", "mmt_first_eos", "mmt_distinct_smiles", "mmt_ingest_peaks", "mmt_ingest_ir", "mmt_sample", "mmt_exponential", "mmt_sample_probs", "mmt_sample_memory_streams", "mmt_sample_controlled", "mmt_linear", "mmt_ffn",
    "mmt_decode_self_attention", "mmt_decode_cross_attention", "mmt_decode_layer_tail", "mmt_encoder_layer", "mmt_launch_count",
    "mmt_profile_enable", "mmt_profile_report",
]

MODE_BITS = {"1H": 1, "13C": 2, "HSQC": 4, "COSY": 8, "IR": 16, "MF": 32, "MS": 64, "MW": 128}
PREC_FP32, PREC_BF16 = 0, 1
SAMPLE_GREEDY, SAMPLE_MULTINOMIAL = 0, 1


class ModelDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "d_model", "n_heads", "n_heads_cross", "d_ff", "n_enc_layers", "n_dec_layers", "vocab",
        "max_len", "mf_vocab", "ms_vocab", "ir_bins", "fp_size", "pad_points")]


class Spectra(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "d_src_1H", "d_mask_1H", "d_src_13C", "d_mask_13C", "d_src_HSQC", "d_mask_HSQC",
        "d_src_COSY", "d_mask_COSY", "d_src_IR", "d_src_MF", "d_mask_MF", "d_src_MS", "d_mask_MS",
        "d_trg_MW")]


class DecodeArgs(C.Structure):
    _fields_ = [
        ("d_memory", C.c_void_p), ("stride_s", C.c_int64), ("stride_b", C.c_int64),
        ("d_key_bias", C.c_void_p), ("S", C.c_int32), ("Bm", C.c_int32), ("n_cand", C.c_int32),
        ("max_len", C.c_int32), ("temperature", C.c_float), ("sampling", C.c_int32),
        ("stop_on_all_pad", C.c_int32), ("precision", C.c_int32),
        ("philox_seed", C.c_uint64), ("philox_offset", C.c_uint64),
        ("seq_index_base", C.c_int64), ("N_total", C.c_int64),
        ("rng_sm_count", C.c_int32), ("rng_max_threads_per_sm", C.c_int32),
    ]


class SamplingControls(C.Structure):
    _fields_ = [("count", C.c_int64), ("h_temperature", C.c_void_p), ("h_top_k", C.c_void_p), ("h_top_p", C.c_void_p)]


def mode_bits(training_mode: str) -> int:
    """Substring tests exactly like the reference ('"1H" in config.training_mode')."""
    bits = 0
    for key, bit in MODE_BITS.items():
        if key in training_mode:
            bits |= bit
    return bits


class NvccMissing(RuntimeError):
    """No compiler on this box (the GPU box runs the .so shipped with the snapshot)."""


def _stale(srcs) -> bool:
    return not os.path.exists(LIB_PATH) or any(os.path.getmtime(LIB_PATH) < os.path.getmtime(s) for s in srcs)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU).

    Safe under torchrun: ranks serialise on a file lock, the compiler writes to a temporary file in the same
    directory and the result is moved into place with an atomic rename, so no process can ever dlopen a
    half-written library; a rank that waited for the lock finds the library fresh and returns."""
    import fcntl
    import tempfile
    srcs = SOURCES + [os.path.join(_HERE, "csrc", f) for f in os.listdir(os.path.join(_HERE, "csrc"))
                      if f.endswith((".cuh", ".h"))] + [HEADER]
    if not force and not _stale(srcs):
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise NvccMissing("nvcc not found: cannot build libmmt_b200.so")
    with open(LIB_PATH + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale(srcs):       # another process built it while this one waited
                return LIB_PATH
            fd, tmp = tempfile.mkstemp(prefix=".libmmt_b200.", suffix=".so.tmp", dir=_HERE)
            os.close(fd)
            try:
                res = subprocess.run([nvcc] + NVCC_FLAGS + ["-o", tmp] + SOURCES, capture_output=True, text=True)
                if res.returncode != 0:
                    raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
                os.chmod(tmp, 0o755)
                os.replace(tmp, LIB_PATH)
            finally:
                if os.path.exists(tmp):
                    os.unlink(tmp)
            if verbose:
                print(res.stdout + res.stderr)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


_LIB = None


def lib():
    """Load (building if sources are newer and nvcc exists) and type the C ABI."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = os.environ.get("MMT_B200_LIB")      # A/B experiments: load another build of the same ABI
    if path:
        if not os.path.exists(path):
            raise RuntimeError(f"MMT_B200_LIB={path} does not exist")
    else:
        path = LIB_PATH
        try:
            build()              # no-op when the library is newer than every source
        except NvccMissing:
            if not os.path.exists(LIB_PATH):
                raise            # nothing shipped and nothing to build it with: fail loudly (no CPU fallback)
            # no compiler on this box: the .so shipped with the snapshot is the build.  Compile errors are NOT swallowed.
    L = C.CDLL(path)
    vp, i32, i64, u64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float
    D = C.POINTER(ModelDesc)
    L.mmt_abi_version.restype = i32
    L.mmt_last_error.restype = C.c_char_p
    L.mmt_weight_count.argtypes = [D]; L.mmt_weight_count.restype = i32
    L.mmt_weight_name.argtypes = [D, i32]; L.mmt_weight_name.restype = C.c_char_p
    L.mmt_weight_numel.argtypes = [D, i32]; L.mmt_weight_numel.restype = i64
    L.mmt_weight_offset.argtypes = [D, i32]; L.mmt_weight_offset.restype = i64
    L.mmt_weight_total.argtypes = [D]; L.mmt_weight_total.restype = i64
    L.mmt_create.argtypes = [D, vp, i64, i32, C.POINTER(vp)]; L.mmt_create.restype = i32
    L.mmt_destroy.argtypes = [vp]; L.mmt_destroy.restype = None
    L.mmt_memory_len.argtypes = [D, C.c_uint32]; L.mmt_memory_len.restype = i32
    L.mmt_mask_is_float.argtypes = [C.c_uint32]; L.mmt_mask_is_float.restype = i32
    L.mmt_encode.argtypes = [vp, C.POINTER(Spectra), i32, C.c_uint32, i32, vp, vp, vp, vp, vp, vp, vp]
    L.mmt_encode.restype = i32
    L.mmt_decode.argtypes = [vp, C.POINTER(DecodeArgs), vp, vp, C.POINTER(i32), vp]; L.mmt_decode.restype = i32
    L.mmt_decode_memory_streams.argtypes = [vp, C.POINTER(DecodeArgs), vp, vp, C.POINTER(i32), vp]; L.mmt_decode_memory_streams.restype = i32
    L.mmt_decode_until_eos.argtypes = [vp, C.POINTER(DecodeArgs), i32, i64, vp, vp, vp, C.POINTER(i32), vp, vp]
    L.mmt_decode_until_eos.restype = i32
    SC = C.POINTER(SamplingControls)
    L.mmt_decode_controlled.argtypes = [vp, C.POINTER(DecodeArgs), i32, i64, SC, vp, vp, vp, C.POINTER(i32), vp, vp]
    L.mmt_decode_controlled.restype = i32
    L.mmt_sample_controlled.argtypes = [vp, vp, vp, i64, i32, SC, i32, i32, i32, u64, u64, i64, i64, i32, i32, vp, vp, vp, vp, vp]
    L.mmt_sample_controlled.restype = i32
    L.mmt_spectra_equal.argtypes = [vp, C.POINTER(Spectra), C.POINTER(Spectra), i32, C.c_uint32, C.POINTER(C.c_int32), vp]; L.mmt_spectra_equal.restype = i32
    L.mmt_teacher_forced.argtypes = [vp, C.POINTER(DecodeArgs), vp, i32, vp, vp]; L.mmt_teacher_forced.restype = i32
    L.mmt_teacher_forced_scores.argtypes = [vp, C.POINTER(DecodeArgs), vp, vp, i32, vp, vp, vp, vp]; L.mmt_teacher_forced_scores.restype = i32
    L.mmt_beam_search.argtypes = [vp, C.POINTER(DecodeArgs), i32, i32, i32, vp, vp, vp, vp, C.POINTER(C.c_int32), vp]; L.mmt_beam_search.restype = i32
    L.mmt_sample_without_replacement.argtypes = [vp, C.POINTER(DecodeArgs), vp, i32, vp, vp, vp, vp, vp, C.POINTER(C.c_int32), vp]
    L.mmt_sample_without_replacement.restype = i32
    L.mmt_sbs_select_step.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp, u64, u64, i64, i32, i32,
                                      vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.mmt_sbs_select_step.restype = i32
    L.mmt_philox_increment.argtypes = [i64, i32, i32]; L.mmt_philox_increment.restype = u64
    L.mmt_pack_tokens_u8.argtypes = [vp, i64, vp, vp]; L.mmt_pack_tokens_u8.restype = i32
    L.mmt_unpack_tokens_u8.argtypes = [vp, i64, vp, vp]; L.mmt_unpack_tokens_u8.restype = i32
    L.mmt_pack_tokens_u8_seqmajor.argtypes = [vp, i32, i64, vp, vp]; L.mmt_pack_tokens_u8_seqmajor.restype = i32
    L.mmt_unpack_tokens_u8_seqmajor.argtypes = [vp, i32, i64, vp, vp]; L.mmt_unpack_tokens_u8_seqmajor.restype = i32
    L.mmt_ingest_peaks.argtypes = [vp, vp, i32, i32, C.c_double, C.c_double, i32, vp, vp, vp]; L.mmt_ingest_peaks.restype = i32
    L.mmt_ingest_ir.argtypes = [vp, vp, i32, i32, vp, vp]; L.mmt_ingest_ir.restype = i32
    L.mmt_first_eos.argtypes = [vp, i32, i64, i32, vp, vp]; L.mmt_first_eos.restype = i32
    L.mmt_sample.argtypes = [vp, vp, i64, f32, i32, u64, u64, i64, i64, i32, i32, vp, vp, vp, vp]
    L.mmt_sample.restype = i32
    L.mmt_exponential.argtypes = [u64, u64, i64, i64, i64, i32, i32, vp, vp]; L.mmt_exponential.restype = i32
    L.mmt_sample_probs.argtypes = [vp, i64, i32, u64, u64, i64, i64, i32, i32, vp, vp]; L.mmt_sample_probs.restype = i32
    L.mmt_sample_memory_streams.argtypes = [vp, vp, vp, i64, i32, i32, i32, f32, u64, u64, i64, i32, i32, vp, vp, vp]
    L.mmt_sample_memory_streams.restype = i32
    L.mmt_distinct_smiles.argtypes = [vp, i32, i64, i32, i64, vp, vp, i32, i32, vp, C.POINTER(i64), C.POINTER(i64), vp]
    L.mmt_distinct_smiles.restype = i32
    L.mmt_linear.argtypes = [vp, vp, vp, vp, vp, i64, i32, i32, i32, i32, vp]; L.mmt_linear.restype = i32
    L.mmt_ffn.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, vp]; L.mmt_ffn.restype = i32
    L.mmt_decode_self_attention.argtypes = [vp, i32, vp, i64, i32, i32, vp, vp]; L.mmt_decode_self_attention.restype = i32
    L.mmt_decode_cross_attention.argtypes = [vp, C.POINTER(DecodeArgs), i32, vp, vp, vp]; L.mmt_decode_cross_attention.restype = i32
    L.mmt_decode_layer_tail.argtypes = [vp, i32, vp, vp, vp, i64, i32, vp, vp, vp, vp, vp]; L.mmt_decode_layer_tail.restype = i32
    L.mmt_encoder_layer.argtypes = [vp, i32, i32, vp, i64, i32, i32, vp, vp, vp, vp, vp, i32, i32, vp, vp, vp, vp]
    L.mmt_encoder_layer.restype = i32
    L.mmt_launch_count.argtypes = [vp]; L.mmt_launch_count.restype = i64
    L.mmt_profile_enable.argtypes = [vp, i32]; L.mmt_profile_enable.restype = i32
    L.mmt_profile_report.argtypes = [vp, C.c_char_p, i64]; L.mmt_profile_report.restype = i32
    if L.mmt_abi_version() != 2:
        raise RuntimeError("libmmt_b200.so ABI version mismatch")
    _LIB = L
    return L


def check(rc: int):
    if rc != 0:
        raise RuntimeError("mmt_b200: " + lib().mmt_last_error().decode("utf-8", "replace"))
