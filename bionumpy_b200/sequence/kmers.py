"""get_kmers / count_kmers (mirror of bionumpy/sequence/kmers.py:36-145).

Hash definition (pinned against the reference's doc goldens): h = sum_j code[i+j] * 4^j, int64,
per-row windows only, rows shorter than k give empty rows.  ``get_kmers`` returns a lazily
materialised EncodedRaggedArray: asking for ``.raw()``/indexing runs the hash kernel (K3);
``count_encoded(kmers, axis=None)`` runs the fused hash+histogram kernel instead and never
writes the hashes."""
import logging

import torch

from .. import _native as nv
from .. import config, ops
from ..encoded_array import EncodedArray, EncodedRaggedArray, BaseEncoding
from ..encodings.alphabet_encoding import AlphabetEncoding, DNAEncoding
from ..encodings.exceptions import EncodingError
from ..encodings.kmer_encodings import KmerEncoding
from ..streams import streamable
from .count_encoded import count_encoded, count_hashed, EncodedCounts

logger = logging.getLogger(__name__)


class _Source:
    """The ragged byte view a lazy value array is computed from."""

    def __init__(self, base, starts, lens, enc_mode, lut, alphabet_encoding, chunk_buffer=None):
        self.base, self.starts, self.lens = base, starts, lens
        self.enc_mode, self.lut, self.alphabet_encoding = enc_mode, lut, alphabet_encoding
        self.chunk_buffer = chunk_buffer     # set when the view is an untouched field of a file buffer


def _source_of(sequence) -> _Source:
    if isinstance(sequence, EncodedArray):
        assert sequence.ndim == 1, "only 1-D EncodedArray and EncodedRaggedArray are supported"
        data = sequence.raw().contiguous()
        starts = torch.zeros(1, dtype=torch.int64, device=data.device)
        lens = torch.full((1,), data.numel(), dtype=torch.int32, device=data.device)
    else:
        data = sequence._data.contiguous()
        starts, lens = sequence._starts.contiguous(), sequence._lens.contiguous()
    if not data.is_cuda:
        raise nv.NativeLibraryError("k-mer kernels need CUDA tensors: bionumpy_b200 has no CPU fallback")
    if data.dtype != torch.uint8:
        data = data.to(torch.uint8)
    enc = sequence.encoding
    if enc.is_base_encoding():
        target = DNAEncoding                                    # kmers.py:70-72
        return _Source(data, starts, lens, target.enc_mode, None, target,
                       getattr(sequence, "_chunk_buffer", None))
    assert isinstance(enc, AlphabetEncoding), \
        "Sequence needs to be encoded with an AlphabetEncoding, e.g. DNAEncoding. " \
        "Change encoding of your sequences by using e.g. bnp.change_encoding(sequences, bnp.DNAEncoding)"
    return _Source(data, starts, lens, nv.ENC_CODES, None, enc)


LONG_ROW = 1 << 14          # rows longer than this are cut into overlapping pieces, one warp each


def _split_long_rows(starts, lens, span, out_offsets=None, piece=LONG_ROW):
    """Rows longer than ``piece`` positions become pieces [i*piece, (i+1)*piece + span - 1): every k-mer /
    window start belongs to exactly one piece, so counts and (with ``out_offsets``) materialised values are
    unchanged while long rows (chromosomes) spread over many warps.  Index arithmetic only (torch);
    returns (starts, lens, out_offsets) of the pieces."""
    L = lens.to(torch.int64)
    if L.numel() == 0 or int(L.max().item()) <= piece + span - 1:
        return starts, lens, out_offsets
    n_pos = torch.clamp(L - (span - 1), min=0)                       # window starts per row
    n_pieces = torch.clamp((n_pos + piece - 1) // piece, min=1)
    row = torch.repeat_interleave(torch.arange(L.numel(), device=L.device), n_pieces)
    first = torch.cumsum(n_pieces, 0) - n_pieces
    idx = torch.arange(row.numel(), device=L.device) - first[row]    # piece index inside its row
    p_start = starts[row] + idx * piece
    p_len = torch.minimum(L[row] - idx * piece, torch.full_like(idx, piece + span - 1))
    p_off = None if out_offsets is None else out_offsets[:-1][row] + idx * piece
    return p_start.contiguous(), p_len.to(torch.int32).contiguous(), p_off


class LazyKmerValues(EncodedRaggedArray):
    """EncodedRaggedArray of k-mer hashes / minimizers whose int64 data appear on first use."""

    def __init__(self, source: _Source, k: int, window_size: int, flat_input: bool = False, canonical: bool = False):
        self._source, self._k, self._window = source, k, window_size
        self._canonical = canonical
        if canonical:
            from .dna import complement_xor_of
            if window_size and source.alphabet_encoding.alphabet_size != 4:
                raise NotImplementedError("minimizers are only implemented for 4-letter alphabets")
            self._cxor = complement_xor_of(source.alphabet_encoding)
        shrink = (window_size if window_size else k) - 1
        self._lens = torch.clamp(source.lens - shrink, min=0).to(torch.int32)
        ends = torch.cumsum(self._lens.to(torch.int64), 0)
        self._starts = ends - self._lens
        self._contiguous = True
        self._encoding = KmerEncoding(source.alphabet_encoding, k)
        self._lazy = None
        self._flat_input = flat_input

    # RaggedArray keeps its flat data in ``_data``; here it is computed on demand
    @property
    def _data(self):
        if self._lazy is None:
            s = self._source
            shrink = (self._window if self._window else self._k) - 1
            if s.alphabet_encoding.alphabet_size != 4:
                # the reference's generic dot-product path (kmers.py:87): plain k-mers only
                if self._window:
                    raise NotImplementedError("minimizers are only implemented for 4-letter alphabets")
                vals, _, status = ops.rows_generic_hash(s.base, s.starts, s.lens, s.alphabet_encoding.alphabet_size,
                                                        self._k, None)
                self._lazy = vals
                return self._lazy
            offsets = ops.row_offsets(s.lens, shrink)
            p_starts, p_lens, p_off = _split_long_rows(s.starts, s.lens, shrink + 1, offsets)
            if p_off is not None and p_off is not offsets:
                total = int(offsets[-1].item())
                p_off = torch.cat([p_off, offsets[-1:]]).contiguous()   # kernels read offsets[row] only
            else:
                total, p_off = None, offsets
            if self._window and self._canonical:
                vals, _, status = ops.rows_minimizers_canonical(s.base, p_starts, p_lens, s.enc_mode, self._k,
                                                                self._window, self._cxor, s.lut, p_off, total=total)
            elif self._window:
                vals, _, status = ops.rows_minimizers(s.base, p_starts, p_lens, s.enc_mode, self._k, self._window,
                                                      s.lut, p_off, total=total)
            elif self._canonical:
                vals, _, status = ops.rows_kmer_hash_canonical(s.base, s.starts, s.lens, s.enc_mode, self._k, self._cxor,
                                                               s.lut, offsets)
                p_starts = s.starts
            else:
                vals, _, status = ops.rows_kmer_hash(s.base, p_starts, p_lens, s.enc_mode, self._k, s.lut, p_off,
                                                     total=total)
            self._check(status, split=p_starts is not s.starts)
            self._lazy = vals
        return self._lazy

    @_data.setter
    def _data(self, v):
        self._lazy = v

    def is_materialised(self):
        return self._lazy is not None

    def _check(self, status, split=False):
        bad = ops.read_status(status).bad_base()
        if bad is not None and split:
            # the (row, position) refers to a piece of a long row: recompute on the unsplit rows (error path)
            s = self._source
            _, status = ops.rows_kmer_count(s.base, s.starts, s.lens, s.enc_mode, 1, 4, 0, s.lut)
            bad = ops.read_status(status).bad_base()
        if bad is not None:
            logging.error("Tried to change encoding of sequences to DNAEncoding, but failed. "
                          "Make sure your sequences are valid DNA, only containing A, C, G, and T")
            self._source.alphabet_encoding._raise_encoding_error(bad[0], bad[1], self._source.lens)

    def fused_histogram(self, n_bins: int) -> torch.Tensor:
        """hist[b] = #{values == b (mod n_bins)} without writing the values (K3/K4 + K5 fused)."""
        s = self._source
        if s.alphabet_encoding.alphabet_size != 4:
            hist, _ = ops.bincount(self._data.contiguous(), n_bins)
            return hist
        buf = s.chunk_buffer
        if buf is not None and buf.can_fuse_count():
            # an untouched sequence field of a file buffer: straight from the raw chunk bytes
            if self._canonical:
                return buf.fused_kmer_histogram(self._k, self._window, n_bins, s.enc_mode, s.lut,
                                                complement_xor=self._cxor)
            return buf.fused_kmer_histogram(self._k, self._window, n_bins, s.enc_mode, s.lut)
        if self._canonical and not self._window:
            hist, status = ops.rows_kmer_count_canonical(s.base, s.starts, s.lens, s.enc_mode, self._k, self._cxor, n_bins, s.lut)
            self._check(status)
            return hist
        span = self._window if self._window else self._k
        p_starts, p_lens, _ = _split_long_rows(s.starts, s.lens, span)
        if self._canonical:
            hist, status = ops.rows_minimizer_count_canonical(s.base, p_starts, p_lens, s.enc_mode, self._k,
                                                              self._window, self._cxor, n_bins, s.lut)
        else:
            hist, status = ops.rows_kmer_count(s.base, p_starts, p_lens, s.enc_mode, self._k, n_bins, self._window,
                                               s.lut)
        self._check(status, split=p_starts is not s.starts)
        return hist


def get_kmers(sequence, k: int, canonical: bool = False):
    """kmers.py:36-87.  ``sequence``: EncodedRaggedArray / 1-D EncodedArray, BaseEncoding text or an
    AlphabetEncoding with four letters; k in 1..31.  EXTENSION: ``canonical=True`` gives min(hash, hash of the
    reverse complement) for every k-mer (sequence/dna.py)."""
    assert 0 < k < 32, "k must be larger than 0 and smaller than 32"
    src = _source_of(sequence)
    out = LazyKmerValues(src, k, 0, canonical=canonical)
    if not config.LAZY:
        out._data
    if isinstance(sequence, EncodedArray):
        return EncodedArray(out._data, out.encoding)
    return out


@streamable(sum)
def count_kmers(sequence, k: int, axis=None) -> EncodedCounts:
    """kmers.py:129-145."""
    return count_encoded(get_kmers(sequence, k), axis=axis)


def count_kmers_hashed(sequence, k: int, n_buckets: int = 1 << 24, window_size: int = 0, canonical: bool = False) -> torch.Tensor:
    """EXTENSION: np.bincount(get_kmers(sequence, k) % n_buckets) (or of the minimizers when
    window_size > 0) as an int64 CUDA tensor, fused.  ``canonical=True`` counts canonical k-mers / minimizers."""
    assert 0 < k < 32, "k must be larger than 0 and smaller than 32"
    assert window_size == 0 or k <= window_size, "kmer size must be smaller than window size"
    return count_hashed(LazyKmerValues(_source_of(sequence), k, window_size, canonical=canonical), n_buckets)
