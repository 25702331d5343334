"""Tensor-level wrappers over the C-ABI (include/bnpk.h).  Everything here runs on the current
CUDA stream of the current device; tensors must be contiguous CUDA tensors.  These are the
operator-level mirror of the reference functions named in include/bnpk.h."""
import ctypes

import torch

from . import _native as nv
from ._native import check, lib, ptr, stream_ptr


def _need_cuda(t, name="tensor"):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise nv.NativeLibraryError(f"{name} must be a CUDA tensor: bionumpy_b200 has no CPU fallback")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")


def _on_device(fn):
    """Run an op with the device of its first tensor argument current (kernels launch on the current device's
    current stream) and check that every tensor argument lives there."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        tensors = [x for x in list(args) + list(kwargs.values()) if isinstance(x, torch.Tensor)]
        dev = next((t.device for t in tensors if t.is_cuda), None)
        if dev is None:
            return fn(*args, **kwargs)
        for t in tensors:
            if t.is_cuda and t.device != dev:
                raise ValueError(f"{fn.__name__}: tensors on different devices ({t.device} and {dev})")
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper


class ScanStatus:
    """Host copy of the device status block (bnpk.h BNPK_ST_*)."""

    def __init__(self, words):
        self.words = [int(w) for w in words]

    n_lines = property(lambda s: s.words[nv.ST_N_LINES])
    n_records = property(lambda s: s.words[nv.ST_N_RECORDS])
    n_complete_bytes = property(lambda s: s.words[nv.ST_N_COMPLETE_BYTES])
    n_bases = property(lambda s: s.words[nv.ST_N_BASES])
    n_values = property(lambda s: s.words[nv.ST_N_VALUES])
    n_long_rows = property(lambda s: s.words[nv.ST_N_LONG_ROWS])
    cr = property(lambda s: bool(s.words[nv.ST_CR]))
    overflow = property(lambda s: bool(s.words[nv.ST_OVERFLOW]))

    @property
    def bad_header_entry(self):
        v = self.words[nv.ST_BAD_HEADER_ENTRY]
        return None if v == nv.INT64_MAX or v >= max(self.n_records, 1) and v != 0 else v

    @property
    def bad_plus_entry(self):
        v = self.words[nv.ST_BAD_PLUS_ENTRY]
        return None if v == nv.INT64_MAX or v >= self.n_records else v

    def bad_base(self, n_rows=None):
        """(row, position) of the first byte outside the alphabet, or None."""
        v = self.words[nv.ST_BAD_BASE]
        if v == nv.INT64_MAX:
            return None
        row, pos = v >> 32, v & 0xFFFFFFFF
        if n_rows is not None and row >= n_rows:
            return None
        return row, pos


def read_status(status_t) -> ScanStatus:
    return ScanStatus(status_t.cpu().tolist())   # synchronises the stream


@_on_device
def count_byte(chunk, value: int) -> int:
    _need_cuda(chunk, "chunk")
    out = torch.empty(1, dtype=torch.int64, device=chunk.device)
    check(lib().bnpk_count_byte(ptr(chunk), chunk.numel(), value, ptr(out), stream_ptr()))
    return int(out.item())


@_on_device
def line_split(chunk, lines_per_entry=4, field_line=1, start_offset=0, header_char=ord("@"), check_plus=True,
               trim_cr=-1, max_rows=None):
    """K1.  Returns (starts int64[R'], lens int32[R'], status tensor).  R' = max_rows (default: the
    exact number of lines / lines_per_entry, obtained with one census pass)."""
    _need_cuda(chunk, "chunk")
    n = chunk.numel()
    dev = chunk.device
    if max_rows is None:
        max_rows = count_byte(chunk, 10) // lines_per_entry
    starts = torch.empty(max_rows, dtype=torch.int64, device=dev)
    lens = torch.empty(max_rows, dtype=torch.int32, device=dev)
    status = nv.new_status(dev)
    ws = nv.workspace(n, dev)
    check(lib().bnpk_line_split(ptr(chunk), n, lines_per_entry, field_line, start_offset, header_char,
                                int(check_plus), trim_cr, ptr(starts), ptr(lens), max_rows, ptr(status),
                                ptr(ws), ws.numel(), stream_ptr()))
    return starts, lens, status


@_on_device
def chunk_kmer_count(chunk, k, n_bins, hist=None, window_size=0, lines_per_entry=4, header_char=ord("@"),
                     check_plus=True, trim_cr=-1, enc_mode=nv.ENC_ASCII_ACGT, lut=None, hist_mode=nv.HIST_AUTO,
                     status=None):
    """K6 on a device-resident chunk.  Accumulates into ``hist`` (int64[n_bins]); returns
    (hist, status tensor)."""
    _need_cuda(chunk, "chunk")
    n = chunk.numel()
    dev = chunk.device
    if hist is None:
        hist = torch.zeros(n_bins, dtype=torch.int64, device=dev)
    if status is None:
        status = nv.new_status(dev)
    ws = nv.workspace(n, dev)
    check(lib().bnpk_chunk_kmer_count(ptr(chunk), n, 0, n, 1, lines_per_entry, header_char, int(check_plus),
                                      trim_cr, enc_mode, ptr(lut), k, window_size, n_bins, hist_mode, ptr(hist),
                                      ptr(status), ptr(ws), ws.numel(), stream_ptr()))
    return hist, status


@_on_device
def chunk_kmer_count_canonical(chunk, k, complement_xor, n_bins, hist=None, lines_per_entry=4, header_char=ord("@"),
                               check_plus=True, trim_cr=-1, enc_mode=nv.ENC_ASCII_ACGT, lut=None, hist_mode=nv.HIST_AUTO,
                               status=None):
    """EXTENSION: K6 on canonical k-mers, min(h, hash of the reverse complement), of a device-resident chunk.
    ``complement_xor``: 3 for ACGT-ordered alphabets, 2 for ACTG.  Accumulates into ``hist`` (int64[n_bins]);
    returns (hist, status tensor)."""
    _need_cuda(chunk, "chunk")
    n = chunk.numel()
    dev = chunk.device
    if hist is None:
        hist = torch.zeros(n_bins, dtype=torch.int64, device=dev)
    if status is None:
        status = nv.new_status(dev)
    ws = nv.workspace(n, dev)
    check(lib().bnpk_chunk_kmer_count_canonical(ptr(chunk), n, 0, n, 1, lines_per_entry, header_char, int(check_plus),
                                                trim_cr, enc_mode, ptr(lut), k, complement_xor, n_bins, hist_mode,
                                                ptr(hist), ptr(status), ptr(ws), ws.numel(), stream_ptr()))
    return hist, status


@_on_device
def chunk_minimizer_count_canonical(chunk, k, window_size, complement_xor, n_bins, hist=None, lines_per_entry=4,
                                    header_char=ord("@"), check_plus=True, trim_cr=-1, enc_mode=nv.ENC_ASCII_ACGT,
                                    lut=None, hist_mode=nv.HIST_AUTO, status=None):
    """EXTENSION: K6 on canonical minimizers, the minimum over each window of ``window_size`` bases of
    min(h, hash of the reverse complement), of a device-resident chunk.  ``complement_xor``: 3 for ACGT-ordered
    alphabets, 2 for ACTG.  Accumulates into ``hist`` (int64[n_bins]); returns (hist, status tensor)."""
    _need_cuda(chunk, "chunk")
    n = chunk.numel()
    dev = chunk.device
    if hist is None:
        hist = torch.zeros(n_bins, dtype=torch.int64, device=dev)
    if status is None:
        status = nv.new_status(dev)
    ws = nv.workspace(n, dev)
    check(lib().bnpk_chunk_minimizer_count_canonical(ptr(chunk), n, 0, n, 1, lines_per_entry, header_char,
                                                     int(check_plus), trim_cr, enc_mode, ptr(lut), k, window_size,
                                                     complement_xor, n_bins, hist_mode, ptr(hist), ptr(status), ptr(ws),
                                                     ws.numel(), stream_ptr()))
    return hist, status


@_on_device
def row_offsets(lens, shrink=0):
    """int64[R+1] exclusive prefix sums of max(lens - shrink, 0)."""
    _need_cuda(lens, "lens")
    if lens.dtype != torch.int32:
        raise TypeError("lens must be int32")
    n = lens.numel()
    out = torch.empty(n + 1, dtype=torch.int64, device=lens.device)
    ws = nv.workspace(max(n, 1), lens.device)
    check(lib().bnpk_row_offsets(ptr(lens), n, shrink, ptr(out), ptr(ws), ws.numel(), stream_ptr()))
    return out


def _rows_args(base, starts, lens):
    _need_cuda(base, "base")
    _need_cuda(starts, "starts")
    _need_cuda(lens, "lens")
    if base.dtype != torch.uint8 or starts.dtype != torch.int64 or lens.dtype != torch.int32:
        raise TypeError("base must be uint8, starts int64, lens int32")
    return ptr(base), base.numel(), ptr(starts), ptr(lens), lens.numel()


@_on_device
def rows_encode(base, starts, lens, enc_mode, lut=None, offsets=None, status=None):
    if offsets is None:
        offsets = row_offsets(lens, 0)
    total = int(offsets[-1].item())
    out = torch.empty(total, dtype=torch.uint8, device=base.device)
    if status is None:
        status = nv.new_status(base.device)
    check(lib().bnpk_rows_encode(*_rows_args(base, starts, lens), enc_mode, ptr(lut), ptr(offsets), ptr(out),
                                 ptr(status), stream_ptr()))
    return out, offsets, status


@_on_device
def rows_kmer_hash(base, starts, lens, enc_mode, k, lut=None, offsets=None, status=None, total=None):
    if offsets is None:
        offsets = row_offsets(lens, k - 1)
    if total is None:
        total = int(offsets[-1].item())
    out = torch.empty(total, dtype=torch.int64, device=base.device)
    if status is None:
        status = nv.new_status(base.device)
    check(lib().bnpk_rows_kmer_hash(*_rows_args(base, starts, lens), enc_mode, ptr(lut), k, ptr(offsets), ptr(out),
                                    ptr(status), stream_ptr()))
    return out, offsets, status


@_on_device
def rows_generic_hash(base, starts, lens, alphabet_size, k, lut=None, offsets=None, status=None):
    """sum_j code[i+j] * alphabet_size^j for alphabets that are not four letters (K3')."""
    if offsets is None:
        offsets = row_offsets(lens, k - 1)
    total = int(offsets[-1].item())
    out = torch.empty(total, dtype=torch.int64, device=base.device)
    if status is None:
        status = nv.new_status(base.device)
    check(lib().bnpk_rows_generic_hash(*_rows_args(base, starts, lens), ptr(lut), alphabet_size, k, ptr(offsets),
                                       ptr(out), ptr(status), stream_ptr()))
    return out, offsets, status


@_on_device
def rows_minimizers(base, starts, lens, enc_mode, k, window_size, lut=None, offsets=None, status=None, total=None):
    if offsets is None:
        offsets = row_offsets(lens, window_size - 1)
    if total is None:
        total = int(offsets[-1].item())
    out = torch.empty(total, dtype=torch.int64, device=base.device)
    if status is None:
        status = nv.new_status(base.device)
    check(lib().bnpk_rows_minimizers(*_rows_args(base, starts, lens), enc_mode, ptr(lut), k, window_size,
                                     ptr(offsets), ptr(out), ptr(status), stream_ptr()))
    return out, offsets, status


@_on_device
def rows_kmer_count(base, starts, lens, enc_mode, k, n_bins, window_size=0, lut=None, hist=None,
                    hist_mode=nv.HIST_AUTO, status=None):
    if hist is None:
        hist = torch.zeros(n_bins, dtype=torch.int64, device=base.device)
    if status is None:
        status = nv.new_status(base.device)
    check(lib().bnpk_rows_kmer_count(*_rows_args(base, starts, lens), enc_mode, ptr(lut), k, window_size, n_bins,
                                     hist_mode, ptr(hist), ptr(status), stream_ptr()))
    return hist, status


@_on_device
@_on_device
def rows_reverse_complement(base, starts, lens, lut, offsets=None):
    """get_reverse_complement on a ragged view: out row r = lut[row r backwards] (uint8, contiguous rows)."""
    if offsets is None:
        offsets = row_offsets(lens, 0)
    total = int(offsets[-1].item())
    out = torch.empty(total, dtype=torch.uint8, device=base.device)
    check(lib().bnpk_rows_reverse_complement(*_rows_args(base, starts, lens), ptr(lut), ptr(offsets), ptr(out), stream_ptr()))
    return out, offsets


@_on_device
def rows_kmer_hash_canonical(base, starts, lens, enc_mode, k, complement_xor, lut=None, offsets=None, status=None):
    """EXTENSION: min(h, hash of the reverse complement) for every k-mer (K3 with a second strand)."""
    if offsets is None:
        offsets = row_offsets(lens, k - 1)
    total = int(offsets[-1].item())
    out = torch.empty(total, dtype=torch.int64, device=base.device)
    if status is None:
        status = nv.new_status(base.device)
    check(lib().bnpk_rows_kmer_hash_canonical(*_rows_args(base, starts, lens), enc_mode, ptr(lut), k, complement_xor,
                                              ptr(offsets), ptr(out), ptr(status), stream_ptr()))
    return out, offsets, status


@_on_device
def rows_kmer_count_canonical(base, starts, lens, enc_mode, k, complement_xor, n_bins, lut=None, hist=None,
                              hist_mode=nv.HIST_AUTO, status=None):
    if hist is None:
        hist = torch.zeros(n_bins, dtype=torch.int64, device=base.device)
    if status is None:
        status = nv.new_status(base.device)
    check(lib().bnpk_rows_kmer_count_canonical(*_rows_args(base, starts, lens), enc_mode, ptr(lut), k, complement_xor,
                                               n_bins, hist_mode, ptr(hist), ptr(status), stream_ptr()))
    return hist, status


@_on_device
def rows_minimizers_canonical(base, starts, lens, enc_mode, k, window_size, complement_xor, lut=None, offsets=None,
                              status=None, total=None):
    """EXTENSION: canonical minimizers, the minimum over each window of min(h, hash of the reverse complement)
    (K4 with a second strand)."""
    if offsets is None:
        offsets = row_offsets(lens, window_size - 1)
    if total is None:
        total = int(offsets[-1].item())
    out = torch.empty(total, dtype=torch.int64, device=base.device)
    if status is None:
        status = nv.new_status(base.device)
    check(lib().bnpk_rows_minimizers_canonical(*_rows_args(base, starts, lens), enc_mode, ptr(lut), k, window_size,
                                               complement_xor, ptr(offsets), ptr(out), ptr(status), stream_ptr()))
    return out, offsets, status


@_on_device
def rows_minimizer_count_canonical(base, starts, lens, enc_mode, k, window_size, complement_xor, n_bins, lut=None,
                                   hist=None, hist_mode=nv.HIST_AUTO, status=None):
    if hist is None:
        hist = torch.zeros(n_bins, dtype=torch.int64, device=base.device)
    if status is None:
        status = nv.new_status(base.device)
    check(lib().bnpk_rows_minimizer_count_canonical(*_rows_args(base, starts, lens), enc_mode, ptr(lut), k,
                                                    window_size, complement_xor, n_bins, hist_mode, ptr(hist),
                                                    ptr(status), stream_ptr()))
    return hist, status


@_on_device
def bincount(values, n_bins, hist=None, hist_mode=nv.HIST_AUTO, status=None):
    _need_cuda(values, "values")
    if values.dtype != torch.int64:
        raise TypeError("values must be int64")
    if hist is None:
        hist = torch.zeros(n_bins, dtype=torch.int64, device=values.device)
    if status is None:
        status = nv.new_status(values.device)
    check(lib().bnpk_bincount(ptr(values), values.numel(), n_bins, hist_mode, ptr(hist), ptr(status), stream_ptr()))
    return hist, status


@_on_device
def bincount_rows(values, offsets, n_bins, status=None):
    _need_cuda(values, "values")
    n_rows = offsets.numel() - 1
    out = torch.zeros((n_rows, n_bins), dtype=torch.int64, device=values.device)
    if status is None:
        status = nv.new_status(values.device)
    check(lib().bnpk_bincount_rows(ptr(values), ptr(offsets), n_rows, n_bins, ptr(out), ptr(status), stream_ptr()))
    return out, status


def synth_fastq(n_records, first_record=0, seed=20240924, device="cuda", out=None):
    """Synthetic 317-byte FASTQ records on the device (bit-identical to the oracle's generator)."""
    if out is None:
        out = torch.empty(n_records * 317, dtype=torch.uint8, device=device)
    check(lib().bnpk_synth_fastq(ptr(out), first_record, n_records, seed, stream_ptr()))
    return out


class HostPipeline:
    """bnpk_pipeline_*: host chunk -> sliced H2D overlapped with the fused count."""

    def __init__(self, capacity_bytes, slice_bytes=64 << 20):
        self._h = ctypes.c_void_p(0)
        check(lib().bnpk_pipeline_create(ctypes.byref(self._h), capacity_bytes, slice_bytes))
        self.capacity = capacity_bytes

    def kmer_count(self, chunk_host, k, hist, window_size=0, lines_per_entry=4, header_char=ord("@"),
                   check_plus=True, trim_cr=-1, enc_mode=nv.ENC_ASCII_ACGT, lut_host=None, hist_mode=nv.HIST_AUTO):
        """chunk_host: CPU uint8 tensor (pinned for real overlap); hist: CUDA int64[n_bins]."""
        if chunk_host.is_cuda or chunk_host.dtype != torch.uint8:
            raise TypeError("chunk_host must be a CPU uint8 tensor")
        status = (ctypes.c_int64 * nv.ST_WORDS)()
        with torch.cuda.device(hist.device):
            check(lib().bnpk_pipeline_kmer_count_host_on(
                self._h, ctypes.c_void_p(chunk_host.data_ptr()), chunk_host.numel(), lines_per_entry, header_char,
                int(check_plus), trim_cr, enc_mode, ctypes.c_void_p(lut_host.data_ptr()) if lut_host is not None else None,
                k, window_size, hist.numel(), hist_mode, ptr(hist), ctypes.cast(status, ctypes.c_void_p), stream_ptr()))
        return ScanStatus(list(status))

    def close(self):
        if self._h:
            nv.load_library().bnpk_pipeline_destroy(self._h)
            self._h = ctypes.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
