"""ctypes binding of libbnpk.so (the C-ABI declared in include/bnpk.h).

There is NO fallback: if the CUDA library is missing or no CUDA device is present, every
compute entry point raises.  The oracle under ``oracle/`` is test infrastructure and is never
imported from here.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libbnpk.so")

# mirror of include/bnpk.h -----------------------------------------------------------------
ENC_ASCII_ACGT, ENC_ASCII_ACTG, ENC_CODES, ENC_LUT = 0, 1, 2, 3
HIST_AUTO, HIST_SMEM, HIST_GLOBAL = 0, 1, 2
E_BADARG, E_K, E_WINDOW, E_WORKSPACE, E_BINS = -1, -2, -3, -4, -5
(ST_N_LINES, ST_N_RECORDS, ST_N_COMPLETE_BYTES, ST_BAD_HEADER_ENTRY, ST_BAD_PLUS_ENTRY, ST_BAD_BASE,
 ST_N_BASES, ST_N_VALUES, ST_N_LONG_ROWS, ST_CR, ST_LAST_ROW_START, ST_LAST_ROW_INDEX, ST_OVERFLOW) = range(13)
ST_WORDS = 16
INT64_MAX = (1 << 63) - 1
SMEM_MAX_BINS = 32768

_vp, _sz, _i, _i64, _u8, _u64 = (ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int64,
                                 ctypes.c_uint8, ctypes.c_uint64)

# name -> (restype, argtypes); tests check every one of these is exported
SIGNATURES = {
    "bnpk_abi_version": (_i, []),
    "bnpk_last_error": (ctypes.c_char_p, []),
    "bnpk_sm_count": (_i, []),
    "bnpk_launch_count": (_u64, []),
    "bnpk_profile_enable": (_i, [_i]),
    "bnpk_profile_read": (_i, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(_u64)]),
    "bnpk_status_init": (_i, [_vp, _vp]),
    "bnpk_count_byte": (_i, [_vp, _sz, _u8, _vp, _vp]),
    "bnpk_tile_workspace_bytes": (_sz, [_sz]),
    "bnpk_tile_workspace_reset": (_i, [_vp, _sz, _vp]),
    "bnpk_line_split": (_i, [_vp, _sz, _i, _i, _i, _u8, _i, _i, _vp, _vp, _sz, _vp, _vp, _sz, _vp]),
    "bnpk_chunk_kmer_count": (_i, [_vp, _sz, _sz, _sz, _i, _i, _u8, _i, _i, _i, _vp, _i, _i, _i64, _i, _vp,
                                   _vp, _vp, _sz, _vp]),
    "bnpk_chunk_kmer_count_canonical": (_i, [_vp, _sz, _sz, _sz, _i, _i, _u8, _i, _i, _i, _vp, _i, _i, _i64, _i, _vp,
                                             _vp, _vp, _sz, _vp]),
    "bnpk_row_offsets": (_i, [_vp, _sz, _i, _vp, _vp, _sz, _vp]),
    "bnpk_rows_encode": (_i, [_vp, _sz, _vp, _vp, _sz, _i, _vp, _vp, _vp, _vp, _vp]),
    "bnpk_rows_kmer_hash": (_i, [_vp, _sz, _vp, _vp, _sz, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "bnpk_rows_generic_hash": (_i, [_vp, _sz, _vp, _vp, _sz, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "bnpk_rows_minimizers": (_i, [_vp, _sz, _vp, _vp, _sz, _i, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "bnpk_rows_kmer_count": (_i, [_vp, _sz, _vp, _vp, _sz, _i, _vp, _i, _i, _i64, _i, _vp, _vp, _vp]),
    "bnpk_rows_reverse_complement": (_i, [_vp, _sz, _vp, _vp, _sz, _vp, _vp, _vp, _vp]),
    "bnpk_rows_kmer_hash_canonical": (_i, [_vp, _sz, _vp, _vp, _sz, _i, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "bnpk_rows_kmer_count_canonical": (_i, [_vp, _sz, _vp, _vp, _sz, _i, _vp, _i, _i, _i64, _i, _vp, _vp, _vp]),
    "bnpk_rows_minimizers_canonical": (_i, [_vp, _sz, _vp, _vp, _sz, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "bnpk_rows_minimizer_count_canonical": (_i, [_vp, _sz, _vp, _vp, _sz, _i, _vp, _i, _i, _i, _i64, _i, _vp, _vp,
                                                 _vp]),
    "bnpk_chunk_minimizer_count_canonical": (_i, [_vp, _sz, _sz, _sz, _i, _i, _u8, _i, _i, _i, _vp, _i, _i, _i, _i64,
                                                  _i, _vp, _vp, _vp, _sz, _vp]),
    "bnpk_bincount": (_i, [_vp, _sz, _i64, _i, _vp, _vp, _vp]),
    "bnpk_bincount_rows": (_i, [_vp, _vp, _sz, _i64, _vp, _vp, _vp]),
    "bnpk_pipeline_create": (_i, [ctypes.POINTER(_vp), _sz, _sz]),
    "bnpk_pipeline_destroy": (None, [_vp]),
    "bnpk_pipeline_kmer_count_host": (_i, [_vp, _vp, _sz, _i, _u8, _i, _i, _i, _vp, _i, _i, _i64, _i, _vp, _vp]),
    "bnpk_pipeline_kmer_count_host_on": (_i, [_vp, _vp, _sz, _i, _u8, _i, _i, _i, _vp, _i, _i, _i64, _i, _vp, _vp, _vp]),
    "bnpk_multiline_flags": (_i, [_vp, _sz, _vp, _vp, _sz, _vp, _vp, _vp]),
    "bnpk_multiline_entries": (_i, [_vp, _vp, _vp, _vp, _vp, _sz, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bnpk_fasta_gather": (_i, [_vp, _sz, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bnpk_bloom_insert": (_i, [_vp, _sz, _vp, _i, _vp, _sz, _vp]),
    "bnpk_bloom_query": (_i, [_vp, _sz, _vp, _i, _vp, _sz, _vp, _vp]),
    "bnpk_synth_fastq": (_i, [_vp, _u64, _u64, _u64, _vp]),
}


class NativeLibraryError(RuntimeError):
    """libbnpk.so is missing / not loadable, or no CUDA device: there is no CPU fallback."""


_lib = None


def load_library(path: str = None):
    """dlopen libbnpk.so and attach prototypes.  Does not need a GPU (used by the CPU tests
    that check the exported symbol list)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise NativeLibraryError(
            f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(bionumpy_b200 has no CPU fallback)")
    try:
        lib = ctypes.CDLL(p)
    except OSError as e:  # pragma: no cover
        raise NativeLibraryError(f"cannot load {p}: {e}") from e
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def lib():
    """The library, for compute: additionally requires a CUDA device."""
    if not torch.cuda.is_available():
        raise NativeLibraryError("bionumpy_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return load_library()


def check(rc: int):
    if rc == 0:
        return
    msg = load_library().bnpk_last_error().decode()
    if rc in (E_K, E_WINDOW):
        raise AssertionError(msg)  # the reference asserts (kmers.py:69, minimizers.py:50)
    if rc < 0:
        raise ValueError(f"bnpk: {msg} (code {rc})")
    raise RuntimeError(f"bnpk: {msg}")


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    if t is None:
        return ctypes.c_void_p(0)
    return ctypes.c_void_p(t.data_ptr())


def new_status(device):
    st = torch.empty(ST_WORDS, dtype=torch.int64, device=device)
    check(lib().bnpk_status_init(ptr(st), stream_ptr()))
    return st


_ws_cache = {}


def workspace(n: int, device):
    """Scratch for the look-back kernels: one buffer per (device, stream), grown on demand.  Two streams never
    share look-back state, and a buffer that is replaced is only freed for the stream that used it (the caching
    allocator reuses a block on its own stream in order)."""
    need = int(load_library().bnpk_tile_workspace_bytes(n))
    with torch.cuda.device(device):
        key = (device.type, device.index if device.index is not None else torch.cuda.current_device(),
               torch.cuda.current_stream().cuda_stream)
        ws = _ws_cache.get(key)
        if ws is None or ws.numel() < need:
            ws = torch.empty(max(need, 1 << 16), dtype=torch.uint8, device=device)
            _ws_cache[key] = ws
    return ws
