"""ctypes binding of libhifigan_b200.so (the C-ABI declared in include/hifigan_b200.h).

There is no fallback: if the shared library is missing and cannot be built with nvcc, importing a
kernel raises.  Nothing here touches `oracle/`.
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import shutil
import subprocess
import threading
import time
from ctypes import POINTER, byref, c_char_p, c_double, c_float, c_int, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libhifigan_b200.so")
SOURCES = ["hg_api.cu", "hg_conv1d_tc.cu", "hg_resblock_pair.cu", "hg_disc.cu", "hg_prep.cu", "hg_mel.cu",
           "hg_wgrad.cu", "hg_train.cu", "hg_batched.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]

_lock = threading.Lock()
_lib = None


class HgError(RuntimeError):
    pass


HASH_PATH = os.path.join(_HERE, "libhifigan_b200.srchash")
_LOCK_PATH = os.path.join(_HERE, ".build.lock")


def _source_hash() -> str:
    """Content hash of everything the library is compiled from (file times do not survive the copy to a GPU box)."""
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    deps = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    deps.append(os.path.join(os.path.dirname(_HERE), "include", "hifigan_b200.h"))
    for d in deps:
        if os.path.isfile(d):
            h.update(os.path.basename(d).encode())
            with open(d, "rb") as f:
                h.update(f.read())
    return h.hexdigest()


def _stale() -> bool:
    if not os.path.exists(LIB_PATH) or not os.path.exists(HASH_PATH):
        return True
    with open(HASH_PATH) as f:
        return f.read().strip() != _source_hash()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every kernel for sm_100a into hifi-gan_b200/libhifigan_b200.so (in-tree).  Safe against several
    processes (torchrun ranks) arriving at once: one compiles into a temporary file under a lock file and renames it
    into place, the others wait for the lock and find the library fresh."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise HgError("nvcc not found: cannot build libhifigan_b200.so")
    deadline = time.time() + 900
    while True:
        try:
            fd = os.open(_LOCK_PATH, os.O_CREAT | os.O_EXCL | os.O_WRONLY)
            os.close(fd)
            break
        except FileExistsError:
            if time.time() > deadline or time.time() - os.path.getmtime(_LOCK_PATH) > 900:
                try:
                    os.unlink(_LOCK_PATH)           # a builder died: take over
                except FileNotFoundError:
                    pass
            time.sleep(0.5)
    try:
        if not force and not _stale():              # somebody else built it while this process waited
            return LIB_PATH
        tmp = LIB_PATH + f".tmp{os.getpid()}"
        cmd = [nvcc] + NVCC_FLAGS + ["-o", tmp] + [os.path.join(CSRC, s) for s in SOURCES]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            if os.path.exists(tmp):
                os.unlink(tmp)
            raise HgError("nvcc failed:\n" + res.stdout + res.stderr)
        if verbose:
            print(res.stderr)
        os.replace(tmp, LIB_PATH)
        with open(HASH_PATH + ".tmp", "w") as f:
            f.write(_source_hash())
        os.replace(HASH_PATH + ".tmp", HASH_PATH)
    finally:
        try:
            os.unlink(_LOCK_PATH)
        except FileNotFoundError:
            pass
    return LIB_PATH


_SIGNATURES = {
    "hg_version": (c_char_p, []),
    "hg_last_error": (c_char_p, []),
    "hg_abi_version": (c_int, []),
    "hg_launch_count": (c_int64, []),
    "hg_timestamp": (c_int, [c_void_p, c_void_p]),
    "hg_pack_conv1d_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hg_convtr1d_geometry": (c_int, [c_int, c_int, c_int, POINTER(c_int), POINTER(c_int)]),
    "hg_pack_convtr1d_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hg_conv1d_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                              c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_float, c_void_p, c_int,
                              c_void_p]),
    "hg_conv1d_fwd_actres": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                     c_void_p, c_float, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_float,
                                     c_void_p, c_int, c_void_p]),
    "hg_conv1d_tap_order": (c_int, [c_int, c_int, c_int, POINTER(c_int)]),
    "hg_conv1d_general_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                      c_int, c_int, c_int, c_void_p, c_float, c_void_p, c_int, c_int, c_void_p]),
    "hg_disc_first_conv_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                       c_int, c_void_p, c_float, c_void_p]),
    "hg_disc_last_conv_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                      c_void_p]),
    "hg_avgpool_4_2_2_fwd": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "hg_disc_export_fmap": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hg_disc_import_fmap": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hg_prep_job_size": (c_int, []),
    "hg_prep_batched": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "hg_resblock_pair_supported": (c_int, [c_int, c_int, c_int]),
    "hg_resblock_single_supported": (c_int, [c_int, c_int, c_int]),
    "hg_resblock_pair_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                     c_int, c_float, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_float,
                                     c_void_p, c_int, c_void_p]),
    "hg_resblock_pair_fwd_actin": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                           c_int, c_int, c_float, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                           c_float, c_void_p, c_int, c_void_p]),
    "hg_float_to_int16": (c_int, [c_void_p, ctypes.c_longlong, c_float, c_void_p, c_void_p]),
    "hg_loss_sum": (c_int, [c_void_p, c_void_p, ctypes.c_longlong, c_int, c_float, c_void_p, c_void_p]),
    "hg_segment_gather": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "hg_segment_stage_i16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hg_segment_stage_mel": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hg_ncl_to_nlc": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p]),
    "hg_nlc_to_ncl": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hg_conv_post_tanh_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hg_mel_plan_create": (c_int, [POINTER(c_void_p), c_int, c_int, c_int, c_int, c_int, c_double, c_double, c_void_p]),
    "hg_mel_plan_destroy": (c_int, [c_void_p]),
    "hg_mel_num_frames": (c_int, [c_void_p, c_int]),
    "hg_mel_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "hg_mel_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "hg_mel_emulate_host": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "hg_mel_bwd_emulate_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "hg_pack_dgrad_weight": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hg_conv1d_dgrad": (c_int, [c_void_p, c_void_p] + [c_int] * 12 + [c_void_p, c_float, c_void_p, c_void_p, c_float,
                                c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_int, c_int,
                                c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "hg_conv1d_wgrad": (c_int, [c_void_p, c_void_p] + [c_int] * 11 + [c_void_p, c_int, c_void_p]),
    "hg_unpack_wgrad_conv": (c_int, [c_void_p] + [c_int] * 7 + [POINTER(c_int), c_void_p, c_void_p]),
    "hg_wgrad_finish_conv": (c_int, [c_void_p] + [c_int] * 7 + [POINTER(c_int), c_void_p, c_void_p, c_int, c_void_p,
                                                                  c_void_p, c_void_p]),
    "hg_wgrad_finish_convtr": (c_int, [c_void_p] + [c_int] * 7 + [c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                                                    c_void_p]),
    "hg_weight_norm_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "hg_fold_weight_norm": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "hg_pack_disc_weight": (c_int, [c_void_p] + [c_int] * 7 + [c_void_p, c_void_p, c_void_p]),
    "hg_spectral_norm_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p]),
    "hg_spectral_norm_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                     c_void_p, c_void_p]),
    "hg_colsum_bf16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hg_conv_post_tanh_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float,
                                      c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p]),
    "hg_disc_last_conv_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float,
                                      c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hg_disc_first_conv_bwd": (c_int, [c_void_p, c_void_p, c_void_p] + [c_int] * 8 + [c_void_p] * 4),
    "hg_avgpool_4_2_2_bwd": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "hg_loss_grad": (c_int, [c_void_p, c_void_p, ctypes.c_longlong, c_int, c_float, c_float, c_float, c_void_p,
                             c_void_p, c_void_p]),
    "hg_adamw_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_longlong, c_float, c_float, c_float,
                              c_float, c_float, c_int, c_void_p, c_void_p, c_float, c_void_p]),
    "hg_grad_norm_slot_size": (c_int, []),
    "hg_grad_sumsq": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, c_void_p]),
    "hg_grad_norm_finalize": (c_int, [c_void_p, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p]),
    "hg_adamw_step_guarded": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_longlong, c_float, c_float,
                                      c_float, c_float, c_float, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                      c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def lib() -> ctypes.CDLL:
    """Load (building first if the .so is missing or older than its sources) and return the typed library handle."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if _stale():                            # missing, or csrc/ / the header changed since it was built
                build()
            handle = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(handle, name)
                fn.restype = res
                fn.argtypes = args
            if handle.hg_abi_version() != 3:
                raise HgError("libhifigan_b200.so ABI mismatch")
            _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().hg_last_error().decode("utf-8", "replace")
        raise HgError(f"{what or 'hifigan_b200'} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(lib().hg_launch_count())
