"""Device-side file buffers honouring the reference's FileBuffer plug-in protocol
(bionumpy/io/file_buffers.py:80-271; docs_source/developer_guide/design_principles.rst:23-31):
``from_raw_buffer`` = one pass of the look-back line census (K1, status only) on the device,
fields are (raw chunk, starts, lens) views produced on demand by K1, and the sequence field of an
untouched buffer can be histogrammed straight from the raw bytes by the fused kernel (K6).

  CudaFastQBuffer          <- FastQBuffer          bionumpy/io/fastq_buffer.py:14-61
  CudaTwoLineFastaBuffer   <- TwoLineFastaBuffer   bionumpy/io/one_line_buffer.py:185-192
  CudaMultiLineFastaBuffer <- MultiLineFastaBuffer bionumpy/io/multiline_buffer.py:15-109
"""
import numpy as np
import torch

from .. import _native as nv
from .. import config, ops
from ..datatypes import SequenceEntry, SequenceEntryWithQuality
from ..encoded_array import EncodedArray, EncodedRaggedArray, BaseEncoding
from ..ragged import RaggedArray
from .exceptions import FormatException, IncompleteEntryException


def _to_device_bytes(chunk):
    if isinstance(chunk, EncodedArray):
        chunk = chunk.raw()
    if isinstance(chunk, np.ndarray):
        chunk = torch.from_numpy(np.array(chunk, dtype=np.uint8, copy=not chunk.flags.writeable))
    if not isinstance(chunk, torch.Tensor):
        chunk = torch.frombuffer(bytearray(chunk), dtype=torch.uint8)
    if not chunk.is_cuda:
        dev = config.default_device()
        if dev.type != "cuda":
            raise nv.NativeLibraryError("file buffers need a CUDA device: bionumpy_b200 has no CPU fallback")
        chunk = chunk.to(dev, non_blocking=True)
    return chunk.contiguous()


class FieldView(EncodedRaggedArray):
    """A field of every entry as a zero-copy (raw chunk, starts, lens) view
    (TextBufferExtractor.get_field_by_number, io/file_buffers.py:315-338)."""

    def __init__(self, data, lens, starts, chunk_buffer=None):
        super().__init__(EncodedArray(data, BaseEncoding), lens, starts=starts)
        self._chunk_buffer = chunk_buffer


class CudaOneLineBuffer:
    n_lines_per_entry = 2
    HEADER = ">"
    _line_offsets = (1, 0)
    _check_plus = False
    dataclass = SequenceEntry
    _field_lines = (0, 1)          # field number -> line of the entry

    def __init__(self, data, n_records, cr):
        self._data = data              # device bytes, complete entries only
        self._n_records = n_records
        self._cr = cr
        self._fields = {}

    # ---- protocol -----------------------------------------------------------------------------
    @classmethod
    def read_header(cls, file_object):
        return None

    @classmethod
    def modify_class_with_header_data(cls, header_data):
        return cls

    @classmethod
    def contains_complete_entry(cls, chunks):
        assert len(chunks) == 1
        try:
            return True, cls.from_raw_buffer(chunks[0])
        except IncompleteEntryException:
            return False

    @classmethod
    def from_raw_buffer(cls, chunk, header_data=None):
        """OneLineBuffer.from_raw_buffer + _validate (io/one_line_buffer.py:44-71,155-173;
        io/fastq_buffer.py:38-45)."""
        assert header_data is None
        chunk = _to_device_bytes(chunk)
        lpe = cls.n_lines_per_entry
        _, _, status = ops.line_split(chunk, lpe, 1, 0, ord(cls.HEADER), cls._check_plus, -1, max_rows=0)
        st = ops.read_status(status)
        if st.n_lines < lpe:
            raise IncompleteEntryException("No complete entry in buffer. Try increasing chunk_size.")
        if st.bad_header_entry is not None:
            raise FormatException(f"Expected header line to start with {cls.HEADER}",
                                  line_number=st.bad_header_entry * lpe)
        if st.bad_plus_entry is not None:
            raise FormatException("Expected '+' at third line of entry", line_number=2 + st.bad_plus_entry * lpe)
        return cls(chunk[: st.n_complete_bytes], st.n_records, st.cr)

    @property
    def size(self) -> int:
        return self._data.numel()

    @property
    def n_lines(self) -> int:
        return self._n_records * self.n_lines_per_entry

    @property
    def data(self):
        return EncodedArray(self._data, BaseEncoding)

    def count_entries(self) -> int:
        return self._n_records

    def __len__(self):
        return self._n_records

    def get_field_by_number(self, i: int, t=None):
        if i not in self._fields:
            line = self._field_lines[i]
            starts, lens, _ = ops.line_split(self._data, self.n_lines_per_entry, line, self._line_offsets[line],
                                             ord(self.HEADER), False, 1 if self._cr else 0,
                                             max_rows=self._n_records)
            self._fields[i] = FieldView(self._data, lens, starts, chunk_buffer=self if i == 1 else None)
        return self._fields[i]

    get_text_field_by_number = get_field_by_number

    def get_data(self):
        return self.dataclass.lazy(self)

    # ---- fused count on the raw bytes (K6) ------------------------------------------------------
    def can_fuse_count(self) -> bool:
        return True

    def fused_kmer_histogram(self, k, window_size, n_bins, enc_mode, lut, complement_xor=0):
        """Histogram of the k-mers (window_size = 0) or minimizers of the sequence lines; complement_xor != 0 counts
        canonical k-mers (min of a k-mer and its reverse complement) / canonical minimizers instead."""
        if complement_xor and window_size:
            hist, status = ops.chunk_minimizer_count_canonical(self._data, k, window_size, complement_xor, n_bins, None,
                                                               self.n_lines_per_entry, ord(self.HEADER), False,
                                                               1 if self._cr else 0, enc_mode, lut)
        elif complement_xor:
            hist, status = ops.chunk_kmer_count_canonical(self._data, k, complement_xor, n_bins, None, self.n_lines_per_entry,
                                                          ord(self.HEADER), False, 1 if self._cr else 0, enc_mode, lut)
        else:
            hist, status = ops.chunk_kmer_count(self._data, k, n_bins, None, window_size, self.n_lines_per_entry,
                                                ord(self.HEADER), False, 1 if self._cr else 0, enc_mode, lut)
        st = ops.read_status(status)
        if st.overflow:
            # pathological line structure (more odd rows than the fused pass keeps scratch for):
            # take the general two-kernel route over the row-offset vector instead
            seq = self.get_field_by_number(1)
            if complement_xor and window_size:
                hist, status = ops.rows_minimizer_count_canonical(seq._data, seq._starts.contiguous(),
                                                                  seq._lens.contiguous(), enc_mode, k, window_size,
                                                                  complement_xor, n_bins, lut)
            elif complement_xor:
                hist, status = ops.rows_kmer_count_canonical(seq._data, seq._starts.contiguous(), seq._lens.contiguous(),
                                                             enc_mode, k, complement_xor, n_bins, lut)
            else:
                hist, status = ops.rows_kmer_count(seq._data, seq._starts.contiguous(), seq._lens.contiguous(), enc_mode,
                                                   k, n_bins, window_size, lut)
            st = ops.read_status(status)
        bad = st.bad_base(self._n_records)
        if bad is not None:
            from ..encodings.alphabet_encoding import DNAEncoding
            DNAEncoding._raise_encoding_error(bad[0], bad[1], self.get_field_by_number(1)._lens)
        return hist


class CudaTwoLineFastaBuffer(CudaOneLineBuffer):
    HEADER = ">"
    n_lines_per_entry = 2
    dataclass = SequenceEntry


class CudaFastQBuffer(CudaOneLineBuffer):
    HEADER = "@"
    n_lines_per_entry = 4
    _line_offsets = (1, 0, 0, 0)
    _check_plus = True
    dataclass = SequenceEntryWithQuality
    _field_lines = (0, 1, 3)       # name, sequence, quality (fastq_buffer.py:21-30)

    def get_field_by_number(self, i: int, t=None):
        if i == 2 and 2 not in self._fields:
            text = super().get_field_by_number(2)
            # QualityEncoding: byte - 33 (encodings/__init__.py:26)
            self._fields[2] = RaggedArray(text.ravel().raw() - 33, text.lengths)
        return super().get_field_by_number(i, t)


FastQBuffer = CudaFastQBuffer
TwoLineFastaBuffer = CudaTwoLineFastaBuffer
