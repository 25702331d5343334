"""get_minimizers (mirror of bionumpy/sequence/minimizers.py:20-54): for every window of
``window_size`` bases the numeric minimum of its window_size-k+1 k-mer hashes; rows get
L-window_size+1 values.  Computed as hash-once + warp-shuffle sliding minimum (K4)."""
from ..encoded_array import EncodedArray
from ..encodings.alphabet_encoding import AlphabetEncoding
from .kmers import LazyKmerValues, _source_of
from .. import config


def get_minimizers(sequence, k: int, window_size: int, canonical: bool = False):
    """EXTENSION: ``canonical=True`` takes the minimum of min(hash, hash of the reverse complement) over each
    window: a read and its reverse complement give the same values, window j of one being window
    L - window_size - j of the other."""
    assert isinstance(sequence.encoding, AlphabetEncoding), \
        "Sequence needs to be encoded with an AlphabetEncoding, e.g. DNAEncoding"
    assert k <= window_size, "kmer size must be smaller than window size"
    assert 0 < k < 32, "k must be larger than 0 and smaller than 32"
    src = _source_of(sequence)
    out = LazyKmerValues(src, k, window_size, canonical=canonical)
    if not config.LAZY:
        out._data
    if isinstance(sequence, EncodedArray):
        return EncodedArray(out._data, out.encoding)
    return out
