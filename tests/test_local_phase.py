"""The warp-specialised count fixes each tile's record phase from the tile's own bytes and labels entries relative to
the tile; the resolve pass turns the labels into entry indices.  These tests compare the ws route (16-byte-aligned
chunk) bit-exactly with the oracle and with the register-staged kernel (the same bytes one byte off alignment), which
still takes the line index from the cross-tile look-back: histogram and every status word except the internal
LAST_ROW_* pair and N_LONG_ROWS (the two kernels stage different halos)."""
import numpy as np
import pytest

from helpers import oracle_hist
from oracle import bnp_oracle as o

from bionumpy_b200 import _native as nv

TILE = 16384
ROW_MAX = 1024
COMPARED = [w for w in range(nv.ST_WORDS) if w not in (nv.ST_N_LONG_ROWS, nv.ST_LAST_ROW_START, nv.ST_LAST_ROW_INDEX)]


@pytest.fixture(scope="module")
def ops():
    from bionumpy_b200 import ops
    return ops


def fastq(rng, n, lo, hi, qual_first=None, cr=False, empty_every=0):
    """FASTQ text; qual_first: None = random quality, '@' / '+' / 'mix' = every quality line starts with that byte."""
    eol = "\r\n" if cr else "\n"
    parts = []
    for r in range(n):
        L = 0 if empty_every and r % empty_every == 0 else int(rng.integers(lo, hi + 1))
        seq = "".join(rng.choice(list("ACGT"), size=L)) if L else ""
        q = [chr(int(x)) for x in rng.integers(33, 74, size=L)]
        if L and qual_first:
            q[0] = qual_first if qual_first != "mix" else "@+"[r % 2]
        parts.append(f"@r{r}{eol}{seq}{eol}+{eol}{''.join(q)}{eol}")
    return np.frombuffer("".join(parts).encode("ascii"), dtype=np.uint8).copy()


def run_both(ops, host, k=21, bins=1 << 14, canonical=False, **kw):
    """(hist, status words) of the ws route and of the register-staged route on the same bytes."""
    import torch
    buf = torch.zeros(host.size + 64, dtype=torch.uint8, device="cuda")
    out = []
    for shift in (0, 1):
        view = buf[shift: shift + host.size]
        view.copy_(torch.from_numpy(host))
        if canonical:
            h, st = ops.chunk_kmer_count_canonical(view, k, 3, bins, **kw)
        else:
            h, st = ops.chunk_kmer_count(view, k, bins, **kw)
        out.append((h.cpu().numpy(), st.cpu().tolist()))
    return out


def same(ops, host, compare_hist=True, **kw):
    (h0, w0), (h1, w1) = run_both(ops, host, **kw)
    assert [w0[i] for i in COMPARED] == [w1[i] for i in COMPARED], (w0, w1)
    assert not compare_hist or np.array_equal(h0, h1)
    return h0, ops.ScanStatus(w0)


def check_oracle(ops, host, k=21, bins=1 << 14, **kw):
    hist, st = same(ops, host, k=k, bins=bins, **kw)
    want, size, n_bases = oracle_hist(host, k, bins)
    assert not st.overflow
    assert (st.n_complete_bytes, st.n_bases) == (size, n_bases)
    assert np.array_equal(hist, want)
    return st


@pytest.mark.gpu
@pytest.mark.parametrize("check_plus", [True, False])
@pytest.mark.parametrize("qual_first", [None, "@", "+", "mix"])
def test_quality_line_starts(ops, qual_first, check_plus):
    host = fastq(np.random.default_rng(1), 3000, 0, 300, qual_first=qual_first)
    check_oracle(ops, host, check_plus=check_plus)


@pytest.mark.gpu
@pytest.mark.parametrize("lo,hi", [(500, 20000), (6000, 9000), (15000, 20000)])
def test_records_around_the_tile_size(ops, lo, hi):
    """Records of 1-40 KiB: tiles without a line start, tiles with one partial record (phase left to the resolve
    pass), with '@' at every quality line and check_plus off as the hardest case."""
    rng = np.random.default_rng(lo)
    for qual_first, check_plus in ((None, True), ("@", False)):
        host = fastq(rng, 60, lo, hi, qual_first=qual_first)
        check_oracle(ops, host, check_plus=check_plus)


@pytest.mark.gpu
def test_rows_at_the_in_tile_limit(ops):
    rng = np.random.default_rng(3)
    for cr in (False, True):
        parts = [fastq(rng, 1, L, L, cr=cr) for L in [ROW_MAX - 1, ROW_MAX, ROW_MAX + 1] * 40]
        check_oracle(ops, np.concatenate(parts))


@pytest.mark.gpu
def test_newlines_at_every_offset_around_a_tile_boundary(ops):
    rng = np.random.default_rng(4)
    body = fastq(rng, 400, 0, 120, empty_every=7)
    for pad in range(0, 40):
        head = np.frombuffer((f"@{'x' * (TILE - 20 + pad)}\nACGT\n+\nIIII\n").encode(), dtype=np.uint8)
        check_oracle(ops, np.concatenate([head, body]))


@pytest.mark.gpu
def test_empty_rows_and_crlf(ops):
    host = fastq(np.random.default_rng(5), 4000, 0, 60, cr=True, empty_every=3)
    check_oracle(ops, host)


@pytest.mark.gpu
def test_two_line_fasta(ops):
    rng = np.random.default_rng(6)
    parts = []
    for r in range(600):
        L = int(rng.integers(0, 700)) if r % 20 else int(rng.integers(10000, 40000))
        parts.append(f">c{r}\n{''.join(rng.choice(list('ACGT'), size=L)) if L else ''}\n")
    host = np.frombuffer("".join(parts).encode(), dtype=np.uint8).copy()
    _, st = same(ops, host, k=21, bins=1 << 14, lines_per_entry=2, header_char=ord(">"), check_plus=False)
    size, starts, lens = o.two_line_fasta_split(host)
    assert not st.overflow and (st.n_records, st.n_complete_bytes, st.n_bases) == (600, size, int(lens[:, 1].sum()))


@pytest.mark.gpu
def test_minimizer_and_canonical_builds(ops):
    rng = np.random.default_rng(7)
    for host in (fastq(rng, 2000, 0, 300, qual_first="@"), fastq(rng, 50, 500, 20000)):
        hist, st = same(ops, host, k=15, bins=1 << 14, window_size=20)
        want, size, _ = oracle_hist(host, 15, 1 << 14, window=20)
        assert not st.overflow and np.array_equal(hist, want)
        hist, st = same(ops, host, k=21, bins=1 << 14, canonical=True)
        assert not st.overflow and st.n_complete_bytes == size


@pytest.mark.gpu
def test_sliced_launches_through_the_host_pipeline(ops):
    import torch
    host = np.concatenate([fastq(np.random.default_rng(8), 40000, 0, 300),
                           fastq(np.random.default_rng(9), 40, 6000, 20000)])
    want, size, n_bases = oracle_hist(host, 21, 1 << 14)
    pipe = ops.HostPipeline(host.size + (1 << 20), slice_bytes=1 << 20)
    hist = torch.zeros(1 << 14, dtype=torch.int64, device="cuda")
    st = pipe.kmer_count(torch.from_numpy(host), 21, hist)
    pipe.close()
    assert not st.overflow and (st.n_complete_bytes, st.n_bases) == (size, n_bases)
    assert np.array_equal(hist.cpu().numpy(), want)


@pytest.mark.gpu
def test_bad_bases_in_many_tiles(ops):
    host = fastq(np.random.default_rng(10), 6000, 50, 300)
    seq_starts = np.flatnonzero(host[:-1] == 10)[0::4] + 1
    for s in seq_starts[200::350]:
        host[s + 5] = ord("N")
    _, st = same(ops, host, compare_hist=False)     # the table of a chunk with bad bases is not defined (it raises)
    assert not st.overflow and st.bad_base() == (200, 5)


@pytest.mark.gpu
def test_malformed_newlines(ops):
    """An inserted or deleted newline: either OVERFLOW is set (the counts are incomplete and the caller takes the row
    route) or every word equals the register-staged kernel's."""
    base = fastq(np.random.default_rng(11), 1500, 20, 200)
    nls = np.flatnonzero(base == 10)
    for i, pos in enumerate(nls[37::97]):
        host = np.delete(base, pos) if i % 2 else np.insert(base, pos, 10)
        for check_plus in (True, False):
            (h0, w0), (h1, w1) = run_both(ops, host, check_plus=check_plus)
            if w0[nv.ST_OVERFLOW]:
                continue
            assert [w0[j] for j in COMPARED] == [w1[j] for j in COMPARED], (i, w0, w1)
            if w0[nv.ST_BAD_BASE] == nv.INT64_MAX:               # with bad bases the table is not defined (it raises)
                assert np.array_equal(h0, h1), i


@pytest.mark.gpu
def test_no_overflow_on_the_bench_chunk(ops):
    chunk = ops.synth_fastq(10_000_000)
    hist, status = ops.chunk_kmer_count(chunk, 31, 1 << 14)
    st = ops.read_status(status)
    assert not st.overflow and st.n_records == 10_000_000
    assert int(hist.sum().item()) == 10_000_000 * 120
    del chunk
