"""Round-2 additions on the GPU, all through the C-ABI / the torch dispatcher ops, checked against the oracle:
reverse complement (sequence/dna.py:36-65), canonical k-mers (extension), TORCH_LIBRARY ops, two streams at once."""
import numpy as np
import pytest
import torch

from oracle import bnp_oracle as oracle
from helpers import make_fastq, oracle_hist

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bnp():
    import bionumpy_b200 as bnp
    return bnp


def _rows(rng, n_rows, max_len=90):
    lens = rng.integers(0, max_len, size=n_rows).astype(np.int64)
    flat = rng.integers(0, 4, size=int(lens.sum())).astype(np.uint8)
    return flat, lens


def test_reverse_complement_doc_values(bnp):
    """sequence/dna.py:49-65 on text and on encoded rows."""
    seqs = bnp.as_encoded_array(["ACGT", "AACG", "", "TTTTG", "N"])
    rc = bnp.get_reverse_complement(seqs)
    assert [r.to_string() for r in rc] == ["ACGT", "CGTT", "", "CAAAA", "N"]
    enc = bnp.as_encoded_array(["ACGT", "AACG", "G"], bnp.DNAEncoding)
    assert [r.to_string() for r in bnp.get_reverse_complement(enc)] == ["ACGT", "CGTT", "C"]
    one = bnp.get_reverse_complement(bnp.as_encoded_array("GATTACA", bnp.DNAEncoding))
    assert one.to_string() == "TGTAATC"


@pytest.mark.parametrize("alphabet", ["ACGT", "ACTG"])
def test_reverse_complement_random_rows_vs_oracle(bnp, alphabet):
    rng = np.random.default_rng(11)
    flat, lens = _rows(rng, 300)
    want = oracle.reverse_complement_rows(flat, lens, alphabet)
    enc = bnp.ACGTEncoding if alphabet == "ACGT" else bnp.ACTGEncoding
    ragged = bnp.EncodedRaggedArray(bnp.EncodedArray(torch.from_numpy(flat).cuda(), enc), lens)
    got = bnp.get_reverse_complement(ragged)
    assert np.array_equal(got.ravel().raw().cpu().numpy(), want)
    assert np.array_equal(got._lens.cpu().numpy(), lens)
    # lower case / unknown bytes of text map to 0, as the reference's ASCII table does (dna.py:29-34)
    text = np.frombuffer(b"ACGTNacgtx", dtype=np.uint8)
    got = bnp.get_reverse_complement(bnp.EncodedArray(torch.from_numpy(text.copy()).cuda(), bnp.BaseEncoding))
    assert np.array_equal(got.raw().cpu().numpy(), oracle.reverse_complement_rows(text, np.array([10]), None))


@pytest.mark.parametrize("k", [1, 3, 16, 31])
@pytest.mark.parametrize("alphabet", ["ACGT", "ACTG"])
def test_canonical_kmers_vs_oracle(bnp, k, alphabet):
    rng = np.random.default_rng(100 + k)
    flat, lens = _rows(rng, 200, max_len=120)
    want, want_lens = oracle.canonical_kmers(flat, lens, k, alphabet)
    enc = bnp.ACGTEncoding if alphabet == "ACGT" else bnp.ACTGEncoding
    ragged = bnp.EncodedRaggedArray(bnp.EncodedArray(torch.from_numpy(flat).cuda(), enc), lens)
    kmers = bnp.get_kmers(ragged, k, canonical=True)
    assert np.array_equal(kmers.raw().ravel().cpu().numpy(), want)
    assert np.array_equal(kmers._lens.cpu().numpy(), want_lens)
    for bins in (1 << 10, 1000003):
        hist = bnp.count_kmers_hashed(ragged, k, bins, canonical=True)
        assert np.array_equal(hist.cpu().numpy(), oracle.count_bucketed_flat(want, bins))


def test_canonical_is_strand_symmetric(bnp):
    """size-independent property: a read and its reverse complement have the same canonical k-mer multiset."""
    rng = np.random.default_rng(5)
    flat, lens = _rows(rng, 2000, max_len=200)
    ragged = bnp.EncodedRaggedArray(bnp.EncodedArray(torch.from_numpy(flat).cuda(), bnp.DNAEncoding), lens)
    a = bnp.count_kmers_hashed(ragged, 21, 1 << 16, canonical=True)
    b = bnp.count_kmers_hashed(bnp.get_reverse_complement(ragged), 21, 1 << 16, canonical=True)
    assert torch.equal(a, b)


def test_torch_dispatcher_ops_match_oracle():
    """TORCH_LIBRARY(bnpk): the same kernels through torch.ops."""
    from bionumpy_b200 import torch_ops, _native as nv
    ops = torch_ops.load()
    rng = np.random.default_rng(3)
    host = make_fastq(rng, 3000, min_len=0, max_len=220, lower_frac=0.1)
    chunk = torch.from_numpy(host).cuda()
    for k, bins, window in ((31, 1 << 14, 0), (5, 4 ** 5, 0), (11, 1 << 20, 0), (7, 1 << 12, 19)):
        hist = torch.zeros(bins, dtype=torch.int64, device="cuda")
        status = ops.chunk_kmer_count(chunk, k, window, hist)
        want, size, n_bases = oracle_hist(host, k, bins, window)
        st = status.cpu().tolist()
        assert st[nv.ST_N_COMPLETE_BYTES] == size and st[nv.ST_N_BASES] == n_bases and st[nv.ST_N_RECORDS] == 3000
        assert np.array_equal(hist.cpu().numpy(), want)
    starts, lens, status = ops.line_split(chunk, 4, 1, 0, ord("@"), True, -1, 3000)
    s_want, l_want = oracle.fastq_split(host)[:2] if False else (None, None)
    offsets = ops.row_offsets(lens, 30)
    total = int(offsets[-1].item())
    hashes, status = ops.rows_kmer_hash(chunk, starts, lens, nv.ENC_ASCII_ACGT, None, 31, 0, 0, offsets, total)
    hist = torch.zeros(1 << 14, dtype=torch.int64, device="cuda")
    ops.bincount(hashes, hist)
    want, _, _ = oracle_hist(host, 31, 1 << 14)
    assert np.array_equal(hist.cpu().numpy(), want)


def test_two_streams_count_concurrently():
    """Stream-ordered and safe to call from several streams at once: every call owns its scratch state."""
    from bionumpy_b200 import torch_ops, ops as cops
    ops = torch_ops.load()
    rng = np.random.default_rng(8)
    hosts = [make_fastq(rng, 20000, min_len=50, max_len=250) for _ in range(2)]
    chunks = [torch.from_numpy(h).cuda() for h in hosts]
    wants = [oracle_hist(h, 31, 1 << 14)[0] for h in hosts]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    hists = [torch.zeros(1 << 14, dtype=torch.int64, device="cuda") for _ in range(2)]
    torch.cuda.synchronize()
    for rep in range(8):                                       # interleaved launches on two streams
        for i in (0, 1):
            with torch.cuda.stream(streams[i]):
                if rep % 2:
                    ops.chunk_kmer_count(chunks[i], 31, 0, hists[i])
                else:
                    cops.chunk_kmer_count(chunks[i], 31, 1 << 14, hist=hists[i])   # ctypes path: workspace per stream
    torch.cuda.synchronize()
    for i in (0, 1):
        assert np.array_equal(hists[i].cpu().numpy(), 8 * wants[i])


def test_two_devices_one_process():
    """cudaFuncAttributeMaxDynamicSharedMemorySize is per device: a second GPU must work from the same thread."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from bionumpy_b200 import ops as cops
    rng = np.random.default_rng(9)
    host = make_fastq(rng, 5000, min_len=50, max_len=250)
    want = oracle_hist(host, 31, 1 << 14)[0]
    for dev in (0, 1):
        chunk = torch.from_numpy(host).to(f"cuda:{dev}")
        hist, status = cops.chunk_kmer_count(chunk, 31, 1 << 14)
        assert np.array_equal(hist.cpu().numpy(), want)


def test_saccer3_whole_genome_k21(bnp, tmp_path):
    """BASELINE configs[3] in miniature on every chromosome of the reference's example_data/sacCer3.fa, each cut to
    its first 50 kbases (tests/golden/sacCer3_sample.fa.gz): multi-line FASTA -> 17 long rows -> k=21 hashes.
    Bucketed histogram (2^24) AND the exact distinct-k-mer table (np.unique) against the oracle (SURVEY 8d)."""
    import gzip
    import os
    raw = gzip.open(os.path.join(os.path.dirname(__file__), "golden", "sacCer3_sample.fa.gz")).read()
    assert len(raw) == 867596
    path = tmp_path / "sacCer3.fa"
    path.write_bytes(raw)
    # oracle: the reference's multi-line split, encode, hash
    whole = np.frombuffer((raw if raw.endswith(b"\n") else raw + b"\n") + b">", dtype=np.uint8)
    size, hs, hl, flat, seq_lens = oracle.multiline_fasta_split(whole)
    assert seq_lens.size == 17 and int(seq_lens.sum()) == 850455
    codes = oracle.encode_flat(flat, oracle.alphabet_lut("ACGT"))
    want_h, want_lens = oracle.get_kmers(codes, seq_lens, 21)
    B = 1 << 24
    want_hist = oracle.count_bucketed_flat(want_h, B)
    # ours, through bnp.open in chunks and as one buffer
    hist = torch.zeros(B, dtype=torch.int64, device="cuda")
    n_entries, n_chunks = 0, 0
    for chunk in bnp.open(str(path)).read_chunks(min_chunk_size=200_000):
        hist += bnp.count_kmers_hashed(chunk.sequence, 21, B)
        n_entries += len(chunk)
        n_chunks += 1
    assert n_entries == 17 and n_chunks > 1
    assert np.array_equal(hist.cpu().numpy(), want_hist)
    chunk = bnp.open(str(path)).read()
    kmers = bnp.get_kmers(bnp.change_encoding(chunk.sequence, bnp.DNAEncoding), 21)
    got_h = kmers.raw().ravel().cpu().numpy()
    assert np.array_equal(kmers._lens.cpu().numpy(), want_lens)
    u_want, c_want = np.unique(want_h, return_counts=True)
    u_got, c_got = np.unique(got_h, return_counts=True)
    assert np.array_equal(u_got, u_want) and np.array_equal(c_got, c_want)


def _bgzf(data, block=60000):
    import struct, zlib
    out = b""
    for i in range(0, len(data), block):
        blk = data[i:i + block]
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        payload = c.compress(blk) + c.flush()
        out += struct.pack("<BBBBIBBHBBHH", 0x1F, 0x8B, 8, 4, 0, 0, 0xFF, 6, 66, 67, 2, len(payload) + 25) + payload + \
            struct.pack("<II", zlib.crc32(blk), len(blk))
    return out + bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


@pytest.mark.parametrize("kind", ["plain", "gzip", "bgzf"])
@pytest.mark.parametrize("min_chunk_size", [50_000, 5_000_000])
def test_open_ingest_paths_count_like_the_oracle(bnp, tmp_path, kind, min_chunk_size):
    """bnp.open(...).read_chunks() through the pinned / prefetching ingest (io/ingest.py): plain file, ordinary gzip,
    BGZF -- same chunks as gzip.open + the generic reader would give, same histogram as the oracle."""
    import gzip
    rng = np.random.default_rng(21)
    host = make_fastq(rng, 6000, min_len=1, max_len=260, trailing_newline=(kind != "plain"))
    data = host.tobytes()
    path = tmp_path / ("reads.fq" if kind == "plain" else "reads.fq.gz")
    path.write_bytes(data if kind == "plain" else gzip.compress(data, 4) if kind == "gzip" else _bgzf(data))
    want, size, n_bases = oracle_hist(np.frombuffer(data if data.endswith(b"\n") else data + b"\n", dtype=np.uint8), 31, 1 << 14)
    hist = torch.zeros(1 << 14, dtype=torch.int64, device="cuda")
    n_rec, n_chunks = 0, 0
    with bnp.open(str(path)) as f:
        for chunk in f.read_chunks(min_chunk_size=min_chunk_size):
            hist += bnp.count_kmers_hashed(chunk.sequence, 31, 1 << 14)
            n_rec += len(chunk)
            n_chunks += 1
    assert n_rec == 6000 and np.array_equal(hist.cpu().numpy(), want)
    assert n_chunks == (1 if min_chunk_size > len(data) else n_chunks) and (min_chunk_size > len(data) or n_chunks > 5)
    # names and qualities still come out of the chunks (the buffer objects are the ordinary ones)
    with bnp.open(str(path)) as f:
        first = f.read_chunk(min_chunk_size=50_000)
    assert first.sequence[0].to_string() == data.split(b"\n")[1].decode()


def test_indexed_fasta_on_saccer3(bnp, tmp_path):
    """io/indexed_fasta.py:61-206 on the sample of the reference's sacCer3.fa: contig lengths, a whole contig, random
    intervals (line ends skipped on the device) against the oracle's restatement; k-mers of the intervals."""
    import gzip
    import os
    raw = gzip.open(os.path.join(os.path.dirname(__file__), "golden", "sacCer3_sample.fa.gz")).read()
    path = tmp_path / "sacCer3.fa"
    path.write_bytes(raw)
    data = np.frombuffer(raw, dtype=np.uint8)
    idx = oracle.fasta_index(data)
    fa = bnp.IndexedFasta(str(path))
    assert fa.get_contig_lengths() == {k: v["rlen"] for k, v in idx.items()} and len(idx) == 17
    assert sum(fa.get_contig_lengths().values()) == 850455
    chrom = fa["chrIII"]
    assert chrom.raw().cpu().numpy().tobytes() == oracle.indexed_fasta_interval(data, idx["chrIII"], 0, idx["chrIII"]["rlen"]).tobytes()
    rng = np.random.default_rng(2)
    names = [c for c in idx if c != "chrM"]      # chrM ends with two short lines: outside what a .fai can describe
    iv = []
    for _ in range(200):
        c = names[int(rng.integers(len(names)))]
        a = int(rng.integers(0, idx[c]["rlen"] - 1))
        b = int(min(idx[c]["rlen"], a + rng.integers(1, 5000)))
        iv.append((c, a, b))
    iv.append(("chrI", 0, 50))
    iv.append(("chrI", 49, 51))
    seqs = fa.get_interval_sequences(iv)
    flat = seqs.ravel().raw().cpu().numpy()
    pos = 0
    for c, a, b in iv:
        want = oracle.indexed_fasta_interval(data, idx[c], a, b)
        assert want.size == b - a and np.array_equal(flat[pos:pos + b - a], want), (c, a, b)
        pos += b - a
    # the intervals go straight into the k-mer path
    upper = bnp.EncodedRaggedArray(bnp.EncodedArray(seqs.ravel().raw(), bnp.BaseEncoding), seqs._lens)
    hist = bnp.count_kmers_hashed(upper, 21, 1 << 16)
    codes = oracle.encode_flat(flat, oracle.alphabet_lut("ACGT"))
    h, _ = oracle.get_kmers(codes, np.array([b - a for _, a, b in iv]), 21)
    assert np.array_equal(hist.cpu().numpy(), oracle.count_bucketed_flat(h, 1 << 16))


def test_kmer_index_and_bloom_filter(bnp):
    """sequence/indexing/kmer_indexing.py:24-55 and sequence/bloom_filter.py:21-42 against the oracle."""
    rng = np.random.default_rng(17)
    flat, lens = _rows(rng, 400, max_len=60)
    ragged = bnp.EncodedRaggedArray(bnp.EncodedArray(torch.from_numpy(flat).cuda(), bnp.DNAEncoding), lens)
    k = 5
    h, hl = oracle.get_kmers(flat, lens, k)
    want = oracle.kmer_index(h, hl)
    index = bnp.KmerIndex.create_index(ragged, k)
    for key in list(want)[:200] + [int(h[0])]:
        assert index.get_indices(key).cpu().tolist() == want[key]
    assert index.get_indices("ACGTA").cpu().tolist() == want.get(sum("ACGT".index(c) * 4 ** j for j, c in enumerate("ACGTA")), [])
    lookup = bnp.KmerLookup.from_sequences(ragged, k)
    some = next(iter(want))
    assert len(lookup.get_sequences(some)) == len(want[some])
    # Bloom filter
    kmers = bnp.get_kmers(ragged, 21)
    hv, _ = oracle.get_kmers(flat, lens, 21)
    offsets = np.random.RandomState(12345).randint(0, 100003, 3)
    bf = bnp.BloomFilter.from_m_and_k(100003, 3)
    bf.insert(kmers)
    mask = oracle.bloom_filter_mask(hv, offsets, 100003)
    assert np.array_equal(bf._mask.cpu().numpy().astype(bool), mask)
    probe = rng.integers(0, 1 << 42, size=5000)
    got = bf[torch.from_numpy(probe).cuda()].cpu().numpy()
    assert np.array_equal(got, oracle.bloom_filter_query(mask, probe, offsets))
    assert bool(bf[kmers.raw().ravel()].all().item())


@pytest.mark.parametrize("k,bins,window", [(31, 1 << 14, 42), (31, 1 << 14, 43), (7, 100, 12), (16, 4096, 20), (3, 64, 3), (31, 1 << 14, 31)])
def test_minimizer_counts_lane_per_row_kernel(bnp, k, bins, window):
    """Minimizer counts (sequence/minimizers.py:8-17,50-54) through the warp-specialised build (windows of up to 12
    k-mers, one lane per row, two-level block minima) and, one k-mer beyond, through the older kernel: ragged rows
    (empty, shorter than the window, longer than a tile), lower case, \\r\\n, a table that is not a power of two."""
    from bionumpy_b200 import ops
    rng = np.random.default_rng(5)
    for chunk in (make_fastq(rng, 700, 0, 400, lower_frac=0.3), make_fastq(rng, 40, 1500, 20000), make_fastq(rng, 3000, 0, 12),
                  make_fastq(rng, 500, 100, 160, cr=True), oracle.synthetic_fastq(3, 4000)):
        want, size, n_bases = oracle_hist(chunk, k, bins, window)
        hist, status = ops.chunk_kmer_count(torch.from_numpy(chunk).cuda(), k, bins, window_size=window)
        st = ops.read_status(status)
        assert st.n_complete_bytes == size and st.n_bases == n_bases and st.n_values == want.sum()
        assert np.array_equal(hist.cpu().numpy(), want)


def test_minimizer_counts_dense_newlines(bnp):
    """Thousands of newlines per tile: the row warp rebuilds the newline list window by window (minimizer build)."""
    from bionumpy_b200 import ops
    rng = np.random.default_rng(22)
    parts = []
    for _ in range(20000):
        L = int(rng.integers(0, 6))
        seq = "".join(rng.choice(list("ACGT"), size=L)) if L else ""
        parts.append(f"@\n{seq}\n+\n{'I' * L}\n")
    chunk = np.frombuffer("".join(parts).encode("ascii"), dtype=np.uint8).copy()
    for k, bins, window in ((1, 4, 2), (2, 16, 4), (2, 1 << 14, 2)):
        want, size, n_bases = oracle_hist(chunk, k, bins, window)
        hist, status = ops.chunk_kmer_count(torch.from_numpy(chunk).cuda(), k, bins, window_size=window)
        st = ops.read_status(status)
        assert (st.n_records, st.n_complete_bytes, st.n_bases) == (20000, size, n_bases)
        assert np.array_equal(hist.cpu().numpy(), want)
