"""Canonical k-mers (min of a k-mer and its reverse complement) counted straight from raw FASTQ / two-line FASTA chunks
by the fused count (bnpk_chunk_kmer_count_canonical, torch.ops.bnpk.chunk_kmer_count_canonical, and the file-buffer
route of count_kmers_hashed / count_encoded with canonical=True).  Bit-exact against the oracle's canonical_kmers."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from helpers import make_fastq
from oracle import bnp_oracle as o

from bionumpy_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CX = {"ACGT": 3, "ACTG": 2}
ENC = {"ACGT": _native.ENC_ASCII_ACGT, "ACTG": _native.ENC_ASCII_ACTG}


# ---- without a GPU ------------------------------------------------------------------------------------------------
def _ctype(param):
    """ctypes type of one C parameter declaration ("const uint8_t *chunk" -> c_void_p)."""
    if "*" in param:
        return ctypes.c_void_p
    return {"size_t": ctypes.c_size_t, "int": ctypes.c_int, "uint8_t": ctypes.c_uint8,
            "int64_t": ctypes.c_int64}[param.split()[0]]


def test_entry_point_exported_with_header_signature():
    text = open(os.path.join(ROOT, "include", "bnpk.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    m = re.search(r"int\s+bnpk_chunk_kmer_count_canonical\s*\((.*?)\)\s*;", text, flags=re.S)
    assert m
    params = [" ".join(p.split()) for p in m.group(1).split(",")]
    assert params[12] == "int complement_xor"
    want = [_ctype(p) for p in params]
    res, args = _native.SIGNATURES["bnpk_chunk_kmer_count_canonical"]
    assert res is ctypes.c_int and args == want
    # the plain entry point with window_size swapped for complement_xor
    assert args == _native.SIGNATURES["bnpk_chunk_kmer_count"][1]
    lib = _native.load_library()
    assert hasattr(lib, "bnpk_chunk_kmer_count_canonical")
    assert lib.bnpk_abi_version() == 2


def test_dispatcher_op_registered():
    import torch
    from bionumpy_b200 import torch_ops
    ops = torch_ops.load()
    assert hasattr(ops, "chunk_kmer_count_canonical")
    schema = str(torch._C._get_schema("bnpk::chunk_kmer_count_canonical", ""))
    assert "Tensor(a!) hist" in schema and "int complement_xor" in schema


@pytest.mark.parametrize("cx", [0, 4, -1])
def test_bad_complement_xor_is_an_argument_error(cx):
    """Checked before any CUDA call, so it holds without a device (null pointers are never touched)."""
    lib = _native.load_library()
    rc = lib.bnpk_chunk_kmer_count_canonical(None, 0, 0, 0, 1, 4, ord("@"), 1, -1, 0, None, 21, cx, 1 << 14, 0,
                                             None, None, None, 0, None)
    assert rc == _native.E_BADARG
    assert "complement_xor" in lib.bnpk_last_error().decode()


def test_canonical_build_is_sm100a_code_without_spills():
    """The canonical build of the warp-specialised kernel (576 threads: at most 112 registers) keeps to its budget."""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([tool, "-res-usage", _native.LIB_PATH], capture_output=True, text=True).stdout
    blocks = out.split(" Function ")
    name = "_ZN4bnpk3wsc14tile_ws_kernelILi0ELi1EEEvNS_8TileArgsE"
    blk = next(b for b in blocks if b.startswith(name))
    assert "sm_100a" in out
    m = re.search(r"REG:(\d+) STACK:(\d+)", blk)
    assert m and int(m.group(1)) <= 112 and int(m.group(2)) == 0, m.group(0) if m else blk[:200]


# ---- GPU ----------------------------------------------------------------------------------------------------------
def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def ops():
    from bionumpy_b200 import ops
    return ops


def canon_oracle(chunk, k, bins, alphabet="ACGT", lpe=4):
    """np.bincount(canonical_kmers(sequence lines of the complete entries) % bins), complete bytes, bases."""
    size, starts, lens = (o.fastq_split if lpe == 4 else o.two_line_fasta_split)(chunk)
    s, ln = starts[:, 1], lens[:, 1]
    codes = o.encode_flat(o.gather_rows(chunk, s, ln), o.alphabet_lut(alphabet))
    vals, _ = o.canonical_kmers(codes, ln, k, alphabet)
    return o.count_bucketed_flat(vals.astype(np.int64), bins), size, int(ln.sum())


def run(ops, chunk, k, bins, alphabet="ACGT", **kw):
    hist, status = ops.chunk_kmer_count_canonical(chunk if hasattr(chunk, "is_cuda") else dev(chunk), k, CX[alphabet],
                                                  bins, enc_mode=ENC[alphabet], **kw)
    return hist.cpu().numpy(), ops.read_status(status)


def check(ops, chunk, k, bins, alphabet="ACGT", lpe=4, **kw):
    want, size, n_bases = canon_oracle(chunk, k, bins, alphabet, lpe)
    got, st = run(ops, chunk, k, bins, alphabet, **kw)
    assert (st.n_complete_bytes, st.n_bases) == (size, n_bases), (k, bins, st.words)
    assert st.bad_base() is None and st.n_values == want.sum()
    assert np.array_equal(got, want), (k, bins)


BINS = [None, 1000, 1 << 10, 1 << 14, 1 << 15, 1 << 20, 1 << 23]     # None: 4^k (small k only)


@pytest.fixture(scope="module")
def ragged_chunk():
    """lower-case bases, '\\r' line ends, empty rows and rows shorter than k"""
    rng = np.random.default_rng(41)
    a = make_fastq(rng, 700, 0, 300, cr=True, lower_frac=0.3)
    return a


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("k", [1, 5, 16, 17, 21, 31])
def test_canonical_chunk_vs_oracle(ops, ragged_chunk, k, bins):
    if bins is None:
        if k > 8:
            pytest.skip("4^k bins: small k only")
        bins = 4 ** k
    check(ops, ragged_chunk, k, bins)


@pytest.mark.gpu
@pytest.mark.parametrize("alphabet", ["ACGT", "ACTG"])
@pytest.mark.parametrize("k,bins", [(5, 4 ** 5), (16, 1 << 14), (17, 1 << 14), (31, 1 << 14), (21, 1000), (31, 1 << 20)])
def test_canonical_chunk_alphabets(ops, alphabet, k, bins):
    rng = np.random.default_rng(43)
    chunk = make_fastq(rng, 500, 0, 260, alphabet=alphabet, lower_frac=0.1)
    check(ops, chunk, k, bins, alphabet)


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n,min_len,max_len", [(50, 3000, 0, 40), (51, 60, 2500, 12000), (52, 300, 1000, 2300)])
@pytest.mark.parametrize("k,bins", [(21, 1 << 14), (31, 1 << 15), (13, 1 << 20), (31, 777)])
def test_canonical_chunk_short_long_and_truncated(ops, seed, n, min_len, max_len, k, bins):
    """Empty rows and rows shorter than k; rows long enough to be deferred; every record cut at its end."""
    chunk = make_fastq(np.random.default_rng(seed), n, min_len, max_len)
    for cut in (0, 1, 35):   # whole; last newline missing; cut inside the last quality line (incomplete record)
        check(ops, chunk[: chunk.size - cut] if cut else chunk, k, bins)


@pytest.mark.gpu
def test_canonical_chunk_incomplete_tail(ops):
    """Every cut of the last record: the sequence line of an incomplete entry is un-counted with canonical values."""
    chunk = make_fastq(np.random.default_rng(5), 20, 30, 60)
    last = int(np.flatnonzero(chunk == 10)[-5]) + 1
    for end in range(last, chunk.size + 1, 3):
        check(ops, chunk[:end], 9, 1 << 14)
        check(ops, chunk[:end], 21, 1 << 20)


@pytest.mark.gpu
def test_canonical_chunk_two_line_fasta(ops):
    import torch
    rng = np.random.default_rng(31)
    parts = []
    for r in range(1200):
        L = int(rng.integers(0, 700)) if r % 50 else int(rng.integers(3000, 9000))
        parts.append(f">contig{r}\n{''.join(rng.choice(list('ACGTacgt'), size=L)) if L else ''}\n")
    chunk = np.frombuffer("".join(parts).encode("ascii"), dtype=np.uint8).copy()
    buf = torch.empty(chunk.size + 16, dtype=torch.uint8, device="cuda")
    for k, bins in ((21, 1 << 14), (4, 256), (31, 1 << 20)):
        for shift in (0, 3):
            view = buf[shift: shift + chunk.size]
            view.copy_(dev(chunk))
            want, size, n_bases = canon_oracle(chunk, k, bins, lpe=2)
            got, st = run(ops, view, k, bins, lines_per_entry=2, header_char=ord(">"), check_plus=False)
            assert (st.n_records, st.n_complete_bytes, st.n_bases) == (1200, size, n_bases), (k, shift)
            assert np.array_equal(got, want), (k, bins, shift)


@pytest.mark.gpu
def test_canonical_chunk_dense_newlines(ops):
    """Tiles with more newlines than the list holds (walked in windows)."""
    rng = np.random.default_rng(21)
    parts = []
    for _ in range(30000):
        L = int(rng.integers(0, 4))
        seq = "".join(rng.choice(list("ACGT"), size=L)) if L else ""
        parts.append(f"@\n{seq}\n+\n{'I' * L}\n")
    chunk = np.frombuffer("".join(parts).encode("ascii"), dtype=np.uint8).copy()
    for k, bins in ((1, 4), (2, 16), (3, 1 << 14), (3, 1 << 15)):
        check(ops, chunk, k, bins)


@pytest.mark.gpu
def test_canonical_chunk_unaligned_pointer(ops):
    """A chunk that does not start on a 16-byte boundary goes to the register-staged kernel."""
    import torch
    n = 20000
    host = o.synthetic_fastq(0, n)
    buf = torch.empty(host.size + 64, dtype=torch.uint8, device="cuda")
    want, size, n_bases = canon_oracle(host, 31, 1 << 14)
    for shift in (0, 1, 7, 33):
        view = buf[shift: shift + host.size]
        view.copy_(dev(host))
        got, st = run(ops, view, 31, 1 << 14)
        assert (st.n_records, st.n_complete_bytes, st.n_bases) == (n, size, n_bases), shift
        assert np.array_equal(got, want), shift


@pytest.mark.gpu
@pytest.mark.parametrize("bins", [1 << 14, 1 << 20])
def test_canonical_chunk_sliced_c_abi(ops, bins):
    """Feeding the resident buffer in slices through the C-ABI gives the single-launch table."""
    import torch
    nv = _native
    rng = np.random.default_rng(7)
    host = make_fastq(rng, 12000, 0, 400)
    chunk = dev(host)
    want, size, _ = canon_oracle(host, 21, bins)
    N = chunk.numel()
    hist = torch.zeros(bins, dtype=torch.int64, device="cuda")
    status = nv.new_status(chunk.device)
    ws = nv.workspace(N, chunk.device)
    step = 32768 * 7
    b = 0
    while b < N:
        e = min(N, b + step)
        nv.check(nv.lib().bnpk_chunk_kmer_count_canonical(nv.ptr(chunk), N, b, e, int(e == N), 4, ord("@"), 1, -1, 0,
                                                           None, 21, 3, bins, 0, nv.ptr(hist), nv.ptr(status),
                                                           nv.ptr(ws), ws.numel(), nv.stream_ptr()))
        b = e
    assert np.array_equal(hist.cpu().numpy(), want)
    assert ops.read_status(status).n_complete_bytes == size


@pytest.mark.gpu
@pytest.mark.parametrize("bins", [1 << 14, 1 << 24])
def test_canonical_chunk_equals_rows_route_1m_reads(ops, bins):
    """1 M synthetic reads: the fused table equals line_split + rows_kmer_count_canonical."""
    n = 1_000_000
    chunk = ops.synth_fastq(n)
    got, status = ops.chunk_kmer_count_canonical(chunk, 31, 3, bins)
    st = ops.read_status(status)
    assert st.n_records == n and st.n_bases == 150 * n and st.n_values == 120 * n
    starts, lens, _ = ops.line_split(chunk)
    want, _ = ops.rows_kmer_count_canonical(chunk, starts, lens, _native.ENC_ASCII_ACGT, 31, 3, bins)
    assert int(got.sum().item()) == 120 * n
    assert bool((got == want).all().item())


def _revcomp_reads(chunk):
    size, starts, lens = o.fastq_split(chunk)
    out = chunk[:size].copy()
    comp = np.zeros(256, dtype=np.uint8)
    for a, b in zip(b"ACGTacgt", b"TGCAtgca"):
        comp[a] = b
    for s, ln in zip(starts[:, 1], lens[:, 1]):
        out[s: s + ln] = comp[chunk[s: s + ln]][::-1]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("k,bins", [(21, 1 << 14), (31, 1 << 20), (15, 1 << 14)])
def test_canonical_chunk_is_strand_symmetric(ops, k, bins):
    chunk = make_fastq(np.random.default_rng(77), 2000, 0, 300, lower_frac=0.2)
    a, _ = run(ops, chunk, k, bins)
    b, _ = run(ops, _revcomp_reads(chunk), k, bins)
    assert np.array_equal(a, b) and a.sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("k,bins", [(5, 1024), (21, 1 << 14), (31, 1 << 20)])
def test_canonical_chunk_bad_base_like_plain(ops, k, bins):
    chunk = make_fastq(np.random.default_rng(3), 100, 50, 90)
    size, starts, lens = o.fastq_split(chunk)
    row, pos = 57, 13
    chunk[starts[row, 1] + pos] = ord("N")
    _, st = run(ops, chunk, k, bins)
    _, plain = ops.chunk_kmer_count(dev(chunk), k, bins)
    assert st.bad_base() == ops.read_status(plain).bad_base() == (row, pos)


@pytest.mark.gpu
def test_canonical_bad_base_raises_encoding_error_like_plain(tmp_path):
    import bionumpy_b200 as bnp
    chunk = make_fastq(np.random.default_rng(3), 100, 50, 90)
    size, starts, lens = o.fastq_split(chunk)
    chunk[starts[57, 1] + 13] = ord("N")
    p = tmp_path / "bad.fq"
    p.write_bytes(chunk.tobytes())
    errors = []
    for canonical in (False, True):
        with pytest.raises(bnp.EncodingError) as e:
            bnp.count_kmers_hashed(bnp.open(str(p)).read().sequence, 21, 1 << 14, canonical=canonical)
        errors.append(e.value.offset)
    assert errors[0] == errors[1] == int(lens[:57, 1].sum()) + 13


@pytest.mark.gpu
@pytest.mark.parametrize("k,bins", [(5, 4 ** 5), (21, 1 << 14), (31, 1 << 24)])
def test_dispatcher_op_equals_ctypes(ops, k, bins):
    import torch
    from bionumpy_b200 import torch_ops
    tops = torch_ops.load()
    chunk = dev(make_fastq(np.random.default_rng(9), 3000, 0, 300, lower_frac=0.1))
    want, _ = ops.chunk_kmer_count_canonical(chunk, k, 3, bins)
    hist = torch.zeros(bins, dtype=torch.int64, device="cuda")
    status = tops.chunk_kmer_count_canonical(chunk, k, 3, hist)
    assert torch.equal(hist, want)
    assert ops.read_status(status).n_values == int(want.sum().item())


@pytest.mark.gpu
@pytest.mark.parametrize("k,bins", [(21, 1 << 14), (31, 1 << 20), (5, None)])
def test_file_buffer_takes_the_fused_route(ops, tmp_path, monkeypatch, k, bins):
    """count_kmers_hashed / count_encoded(get_kmers) with canonical=True on a bnp.open buffer run the fused count
    (the rows route is made to fail) and give the rows-route table."""
    import bionumpy_b200 as bnp
    from bionumpy_b200 import ops as ops_mod
    chunk = make_fastq(np.random.default_rng(13), 3000, 0, 300, lower_frac=0.1)
    p = tmp_path / "reads.fq"
    p.write_bytes(chunk.tobytes())
    B = bins or 4 ** k
    size, starts, lens = o.fastq_split(chunk)
    seqs = bnp.open(str(p)).read().sequence
    rows_route, _ = ops.rows_kmer_count_canonical(seqs._data, seqs._starts.contiguous(), seqs._lens.contiguous(),
                                                  _native.ENC_ASCII_ACGT, k, 3, B)
    want, _, _ = canon_oracle(chunk, k, B)
    assert np.array_equal(rows_route.cpu().numpy(), want)

    def no_rows_route(*a, **kw):
        raise AssertionError("canonical count of a file buffer took the rows route")
    monkeypatch.setattr(ops_mod, "rows_kmer_count_canonical", no_rows_route)
    seqs = bnp.open(str(p)).read().sequence
    if bins:
        got = bnp.count_kmers_hashed(seqs, k, B, canonical=True)
    else:
        got = bnp.count_encoded(bnp.get_kmers(seqs, k, canonical=True), axis=None).counts
    assert np.array_equal(got.cpu().numpy(), want)
