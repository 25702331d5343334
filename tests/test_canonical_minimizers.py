"""Canonical minimizers: the minimum over each window of min(k-mer, its reverse complement), on every layer -- the row
kernels (bnpk_rows_minimizers_canonical, bnpk_rows_minimizer_count_canonical), the fused chunk count
(bnpk_chunk_minimizer_count_canonical: the wsmc build of the warp-specialised kernel, or the register-staged kernel),
the dispatcher ops and get_minimizers / count_kmers_hashed with canonical=True.  Bit-exact against the oracle below,
which is built from the reference oracle's canonical_kmers and checked against a dot-product brute force."""
import ctypes
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from helpers import make_fastq
from oracle import bnp_oracle as o

from bionumpy_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CX = {"ACGT": 3, "ACTG": 2}
ENC = {"ACGT": _native.ENC_ASCII_ACGT, "ACTG": _native.ENC_ASCII_ACTG}
NEW_ENTRY_POINTS = ("bnpk_rows_minimizers_canonical", "bnpk_rows_minimizer_count_canonical",
                    "bnpk_chunk_minimizer_count_canonical")


# ---- oracle -------------------------------------------------------------------------------------------------------
def canonical_minimizers(codes_flat, lens, k, window_size, alphabet="ACGT"):
    """Per row, the sliding minimum over window_size-k+1 consecutive canonical k-mers (o.canonical_kmers); rows get
    L-window_size+1 values.  Returns (values, lens) as o.get_minimizers does."""
    assert 0 < k <= window_size
    W = window_size - k + 1
    vals, klens = o.canonical_kmers(codes_flat, lens, k, alphabet)
    klens = np.asarray(klens, dtype=np.int64)
    out_lens = np.maximum(klens - (W - 1), 0)
    if vals.size < W or out_lens.sum() == 0:
        return np.zeros(0, dtype=np.int64), out_lens
    mins = np.lib.stride_tricks.sliding_window_view(vals, W).min(axis=-1)
    return mins[o.ragged_indices(np.cumsum(klens) - klens, out_lens)].astype(np.int64), out_lens


def canonical_minimizers_bruteforce(codes_flat, lens, k, window_size, alphabet="ACGT"):
    """Window by window: min over its k-mers of min(dot product of the k-mer, dot product of its reverse complement).
    Small inputs only."""
    comp = o.complement_table(alphabet)
    conv = 4 ** np.arange(k, dtype=np.int64)
    out, out_lens, pos = [], [], 0
    for L in np.asarray(lens, dtype=np.int64):
        row = codes_flat[pos:pos + L].astype(np.int64)
        pos += L
        n = max(L - window_size + 1, 0)
        for j in range(n):
            best = None
            for i in range(j, j + window_size - k + 1):
                km = row[i:i + k]
                v = min(int(km.dot(conv)), int(comp[km][::-1].astype(np.int64).dot(conv)))
                best = v if best is None else min(best, v)
            out.append(best)
        out_lens.append(n)
    return np.array(out, dtype=np.int64), np.array(out_lens, dtype=np.int64)


def random_rows(rng, n_rows, max_len):
    lens = rng.integers(0, max_len + 1, size=n_rows).astype(np.int64)
    return rng.integers(0, 4, size=int(lens.sum())).astype(np.uint8), lens


def rows_of(flat, lens):
    pos = np.concatenate([[0], np.cumsum(lens)])
    return [flat[pos[i]:pos[i + 1]] for i in range(len(lens))]


# ---- without a GPU ------------------------------------------------------------------------------------------------
def _ctype(param):
    """ctypes type of one C parameter declaration ("const uint8_t *chunk" -> c_void_p)."""
    if "*" in param:
        return ctypes.c_void_p
    return {"size_t": ctypes.c_size_t, "int": ctypes.c_int, "uint8_t": ctypes.c_uint8,
            "int64_t": ctypes.c_int64}[param.split()[0]]


@pytest.mark.parametrize("name", NEW_ENTRY_POINTS)
def test_entry_points_exported_with_header_signatures(name):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bnpk.h")).read(), flags=re.S)
    m = re.search(r"int\s+" + name + r"\s*\((.*?)\)\s*;", text, flags=re.S)
    assert m
    params = [" ".join(p.split()) for p in m.group(1).split(",")]
    assert "int window_size" in params and params[params.index("int window_size") + 1] == "int complement_xor"
    res, args = _native.SIGNATURES[name]
    assert res is ctypes.c_int and args == [_ctype(p) for p in params]
    lib = _native.load_library()
    assert hasattr(lib, name)
    assert lib.bnpk_abi_version() == 2


def _call_with_nulls(name, k, window_size, cx):
    lib = _native.load_library()
    if name == "bnpk_rows_minimizers_canonical":
        return lib.bnpk_rows_minimizers_canonical(None, 0, None, None, 1, 0, None, k, window_size, cx, None, None, None,
                                                  None)
    if name == "bnpk_rows_minimizer_count_canonical":
        return lib.bnpk_rows_minimizer_count_canonical(None, 0, None, None, 1, 0, None, k, window_size, cx, 1 << 14, 0,
                                                       None, None, None)
    return lib.bnpk_chunk_minimizer_count_canonical(None, 0, 0, 0, 1, 4, ord("@"), 1, -1, 0, None, k, window_size, cx,
                                                    1 << 14, 0, None, None, None, 0, None)


@pytest.mark.parametrize("name", NEW_ENTRY_POINTS)
@pytest.mark.parametrize("k,window_size,cx,want", [
    (21, 31, 0, _native.E_BADARG), (21, 31, 4, _native.E_BADARG),
    (21, 20, 3, _native.E_WINDOW), (5, 0, 3, _native.E_WINDOW), (5, 1025, 2, _native.E_WINDOW),
    (32, 41, 3, _native.E_K), (0, 41, 3, _native.E_K)])
def test_argument_errors_before_any_cuda_call(name, k, window_size, cx, want):
    """Checked before any CUDA call, so they hold without a device (the null pointers are never touched)."""
    assert _call_with_nulls(name, k, window_size, cx) == want


def _cta_threads(elf_text, func):
    """The CTA size the build was compiled for (EIATTR_MAX_THREADS of the kernel's .nv.info section)."""
    sec = elf_text.split("\n.nv.info." + func + "\n", 1)[1].split("\n\n", 1)[0]
    m = re.search(r"EIATTR_MAX_THREADS\s+Format:\s+\S+\s+Value:\s+(0x[0-9a-f]+)", sec)
    assert m, sec[:400]
    return int(m.group(1), 16)


def test_wsmc_build_is_sm100a_code_within_its_register_budget():
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    res = subprocess.run([tool, "-res-usage", _native.LIB_PATH], capture_output=True, text=True).stdout
    elf = subprocess.run([tool, "-elf", _native.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in res
    for enc in range(4):
        func = f"_ZN4bnpk4wsmc14tile_ws_kernelILi{enc}ELi1EEEvNS_8TileArgsE"
        blk = next(b for b in res.split(" Function ") if b.startswith(func))
        m = re.search(r"REG:(\d+) STACK:(\d+)", blk)
        threads = _cta_threads(elf, func)
        # 64 K registers = four sub-partitions of 16 K; a CTA's warps are spread over them, 8-register granularity
        warps = -(-threads // 32)
        warps_per_smsp = -(-warps // 4)
        budget = (16384 // (warps_per_smsp * 32)) // 8 * 8
        assert m and int(m.group(1)) <= budget and int(m.group(2)) == 0, (func, threads, budget, m.group(0))


def test_dispatcher_op_registered():
    import torch
    from bionumpy_b200 import torch_ops
    tops = torch_ops.load()
    assert hasattr(tops, "chunk_minimizer_count_canonical")
    schema = str(torch._C._get_schema("bnpk::chunk_minimizer_count_canonical", ""))
    assert "Tensor(a!) hist" in schema and "int window_size" in schema and "int complement_xor" in schema


@pytest.mark.parametrize("alphabet", ["ACGT", "ACTG"])
@pytest.mark.parametrize("k,window_size", [(1, 1), (1, 4), (2, 5), (3, 3), (4, 9), (5, 16), (7, 8)])
def test_oracle_equals_bruteforce(alphabet, k, window_size):
    codes, lens = random_rows(np.random.default_rng(k * 100 + window_size), 30, 40)
    got, got_lens = canonical_minimizers(codes, lens, k, window_size, alphabet)
    want, want_lens = canonical_minimizers_bruteforce(codes, lens, k, window_size, alphabet)
    assert np.array_equal(got_lens, want_lens) and np.array_equal(got, want)


@pytest.mark.parametrize("k", [1, 4, 15, 31])
def test_oracle_window_of_one_kmer_is_canonical_kmers(k):
    codes, lens = random_rows(np.random.default_rng(k), 200, 120)
    got, got_lens = canonical_minimizers(codes, lens, k, k)
    want, want_lens = o.canonical_kmers(codes, lens, k)
    assert np.array_equal(got_lens, want_lens) and np.array_equal(got, want)


@pytest.mark.parametrize("alphabet", ["ACGT", "ACTG"])
@pytest.mark.parametrize("k,window_size", [(1, 3), (5, 11), (15, 25), (31, 41), (21, 84)])
def test_oracle_is_strand_symmetric(alphabet, k, window_size):
    """Window j of a row is window L - window_size - j of its reverse complement."""
    codes, lens = random_rows(np.random.default_rng(window_size), 150, 200)
    a, a_lens = canonical_minimizers(codes, lens, k, window_size, alphabet)
    b, b_lens = canonical_minimizers(o.reverse_complement_rows(codes, lens, alphabet), lens, k, window_size, alphabet)
    assert np.array_equal(a_lens, b_lens)
    for ra, rb in zip(rows_of(a, a_lens), rows_of(b, b_lens)):
        assert np.array_equal(ra, rb[::-1])


@pytest.mark.parametrize("k,window_size", [(3, 7), (15, 25), (31, 41)])
def test_oracle_never_above_plain_minimizer(k, window_size):
    codes, lens = random_rows(np.random.default_rng(3), 150, 200)
    canon, c_lens = canonical_minimizers(codes, lens, k, window_size)
    plain, p_lens = o.get_minimizers(codes, lens, k, window_size)
    assert np.array_equal(c_lens, p_lens) and canon.size > 0
    assert (canon <= plain).all() and (canon < plain).any()


# ---- GPU ----------------------------------------------------------------------------------------------------------
def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def ops():
    from bionumpy_b200 import ops
    return ops


def chunk_oracle(chunk, k, window_size, bins, alphabet="ACGT", lpe=4):
    """np.bincount(canonical minimizers of the complete entries' sequence lines % bins), complete bytes, bases."""
    size, starts, lens = (o.fastq_split if lpe == 4 else o.two_line_fasta_split)(chunk)
    s, ln = starts[:, 1], lens[:, 1]
    codes = o.encode_flat(o.gather_rows(chunk, s, ln), o.alphabet_lut(alphabet))
    vals, _ = canonical_minimizers(codes, ln, k, window_size, alphabet)
    return o.count_bucketed_flat(vals, bins), size, int(ln.sum())


def run(ops, chunk, k, window_size, bins, alphabet="ACGT", lut=False, **kw):
    if lut:
        kw.update(enc_mode=_native.ENC_LUT, lut=dev(o.alphabet_lut(alphabet)))
    else:
        kw.setdefault("enc_mode", ENC[alphabet])
    hist, status = ops.chunk_minimizer_count_canonical(chunk if hasattr(chunk, "is_cuda") else dev(chunk), k,
                                                       window_size, CX[alphabet], bins, **kw)
    return hist.cpu().numpy(), ops.read_status(status)


def check(ops, chunk, k, window_size, bins, alphabet="ACGT", lpe=4, **kw):
    want, size, n_bases = chunk_oracle(chunk, k, window_size, bins, alphabet, lpe)
    got, st = run(ops, chunk, k, window_size, bins, alphabet, **kw)
    assert (st.n_complete_bytes, st.n_bases) == (size, n_bases), (k, window_size, bins, st.words)
    assert st.bad_base() is None and st.n_values == want.sum()
    assert np.array_equal(got, want), (k, window_size, bins)


# W = k-mers per window: 1..12 go to the wsmc build (CTA-private tables), 13.. to the register-staged kernel
KS = [1, 5, 15, 16, 17, 21, 31]
WS = [1, 2, 11, 12, 13, 32, 33, 64]
BINS = [None, 1000, 1 << 10, 1 << 14, 1 << 15, 1 << 20, 1 << 23]     # None: 4^k (small k only)


@pytest.fixture(scope="module")
def ragged_chunk():
    """lower-case bases, '\\r' line ends, empty rows and rows shorter than the window"""
    return make_fastq(np.random.default_rng(41), 700, 0, 300, cr=True, lower_frac=0.3)


@pytest.mark.gpu
@pytest.mark.parametrize("W", WS)
@pytest.mark.parametrize("k", KS)
def test_fused_count_vs_oracle(ops, ragged_chunk, k, W):
    check(ops, ragged_chunk, k, k + W - 1, 1 << 14)


@pytest.mark.gpu
@pytest.mark.parametrize("bins", BINS)
@pytest.mark.parametrize("k,W", [(1, 2), (5, 12), (15, 11), (17, 1), (31, 12), (16, 33), (31, 64)])
def test_fused_count_bins(ops, ragged_chunk, k, W, bins):
    if bins is None:
        if k > 8:
            pytest.skip("4^k bins: small k only")
        bins = 4 ** k
    check(ops, ragged_chunk, k, k + W - 1, bins)


@pytest.mark.gpu
@pytest.mark.parametrize("lut", [False, True])
@pytest.mark.parametrize("alphabet", ["ACGT", "ACTG"])
@pytest.mark.parametrize("k,W,bins", [(5, 4, 4 ** 5), (15, 11, 1 << 14), (31, 12, 1000), (17, 32, 1 << 14),
                                      (21, 12, 1 << 20)])
def test_fused_count_alphabets_and_lut(ops, alphabet, lut, k, W, bins):
    chunk = make_fastq(np.random.default_rng(43), 500, 0, 260, alphabet=alphabet, lower_frac=0.1)
    check(ops, chunk, k, k + W - 1, bins, alphabet, lut=lut)


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n,min_len,max_len", [(50, 3000, 0, 40), (51, 60, 2500, 12000), (52, 300, 1000, 2300)])
@pytest.mark.parametrize("k,W,bins", [(21, 12, 1 << 14), (31, 33, 1 << 15), (15, 2, 1 << 20), (31, 11, 777)])
def test_fused_count_short_long_and_truncated(ops, seed, n, min_len, max_len, k, W, bins):
    """Rows shorter than the window; rows longer than the tile halo (deferred list); every record cut at its end."""
    chunk = make_fastq(np.random.default_rng(seed), n, min_len, max_len)
    for cut in (0, 1, 35):   # whole; last newline missing; cut inside the last quality line (incomplete record)
        check(ops, chunk[: chunk.size - cut] if cut else chunk, k, k + W - 1, bins)


@pytest.mark.gpu
def test_fused_count_incomplete_tail(ops):
    """Every cut of the last record: the sequence line of an incomplete entry is un-counted with canonical values."""
    chunk = make_fastq(np.random.default_rng(5), 20, 30, 60)
    last = int(np.flatnonzero(chunk == 10)[-5]) + 1
    for end in range(last, chunk.size + 1, 3):
        check(ops, chunk[:end], 9, 19, 1 << 14)
        check(ops, chunk[:end], 21, 41, 1 << 20)


@pytest.mark.gpu
def test_fused_count_two_line_fasta(ops):
    import torch
    rng = np.random.default_rng(31)
    parts = []
    for r in range(1200):
        L = int(rng.integers(0, 700)) if r % 50 else int(rng.integers(3000, 9000))
        parts.append(f">contig{r}\n{''.join(rng.choice(list('ACGTacgt'), size=L)) if L else ''}\n")
    chunk = np.frombuffer("".join(parts).encode("ascii"), dtype=np.uint8).copy()
    buf = torch.empty(chunk.size + 16, dtype=torch.uint8, device="cuda")
    for k, w, bins in ((21, 31, 1 << 14), (4, 6, 256), (31, 80, 1 << 20)):
        for shift in (0, 3):
            view = buf[shift: shift + chunk.size]
            view.copy_(dev(chunk))
            want, size, n_bases = chunk_oracle(chunk, k, w, bins, lpe=2)
            got, st = run(ops, view, k, w, bins, lines_per_entry=2, header_char=ord(">"), check_plus=False)
            assert (st.n_records, st.n_complete_bytes, st.n_bases) == (1200, size, n_bases), (k, shift)
            assert np.array_equal(got, want), (k, bins, shift)


@pytest.mark.gpu
def test_fused_count_dense_newlines(ops):
    """Tiles with more newlines than the list holds (walked in windows)."""
    rng = np.random.default_rng(21)
    parts = []
    for _ in range(30000):
        L = int(rng.integers(0, 6))
        seq = "".join(rng.choice(list("ACGT"), size=L)) if L else ""
        parts.append(f"@\n{seq}\n+\n{'I' * L}\n")
    chunk = np.frombuffer("".join(parts).encode("ascii"), dtype=np.uint8).copy()
    for k, w, bins in ((1, 1, 4), (1, 3, 4), (2, 4, 16), (3, 5, 1 << 14), (3, 5, 1 << 15)):
        check(ops, chunk, k, w, bins)


@pytest.mark.gpu
def test_fused_count_unaligned_pointer(ops):
    """A chunk that does not start on a 16-byte boundary goes to the register-staged kernel."""
    import torch
    n = 20000
    host = o.synthetic_fastq(0, n)
    buf = torch.empty(host.size + 64, dtype=torch.uint8, device="cuda")
    want, size, n_bases = chunk_oracle(host, 31, 41, 1 << 14)
    for shift in (0, 1, 7, 33):
        view = buf[shift: shift + host.size]
        view.copy_(dev(host))
        got, st = run(ops, view, 31, 41, 1 << 14)
        assert (st.n_records, st.n_complete_bytes, st.n_bases) == (n, size, n_bases), shift
        assert np.array_equal(got, want), shift


@pytest.mark.gpu
@pytest.mark.parametrize("k,w,bins", [(21, 31, 1 << 14), (15, 60, 1 << 14), (21, 31, 1 << 20)])
def test_fused_count_sliced_c_abi(ops, k, w, bins):
    """Feeding the resident buffer in slices through the C-ABI gives the single-launch table."""
    import torch
    nv = _native
    host = make_fastq(np.random.default_rng(7), 12000, 0, 400)
    chunk = dev(host)
    want, size, _ = chunk_oracle(host, k, w, bins)
    N = chunk.numel()
    hist = torch.zeros(bins, dtype=torch.int64, device="cuda")
    status = nv.new_status(chunk.device)
    ws = nv.workspace(N, chunk.device)
    step = 32768 * 7
    b = 0
    while b < N:
        e = min(N, b + step)
        nv.check(nv.lib().bnpk_chunk_minimizer_count_canonical(nv.ptr(chunk), N, b, e, int(e == N), 4, ord("@"), 1, -1,
                                                                0, None, k, w, 3, bins, 0, nv.ptr(hist),
                                                                nv.ptr(status), nv.ptr(ws), ws.numel(), nv.stream_ptr()))
        b = e
    assert np.array_equal(hist.cpu().numpy(), want)
    assert ops.read_status(status).n_complete_bytes == size


_REG_SCRIPT = """
import sys
import numpy as np
import torch
from bionumpy_b200 import ops
chunk = torch.from_numpy(np.load(sys.argv[1])).cuda()
out = [ops.chunk_minimizer_count_canonical(chunk, k, w, 3, bins)[0].cpu().numpy()
       for k, w, bins in ((31, 41, 1 << 14), (15, 25, 1 << 14), (21, 60, 1 << 20))]
np.save(sys.argv[2], np.concatenate(out))
"""


@pytest.mark.gpu
def test_register_staged_kernel_gives_the_same_tables(ops, tmp_path):
    """BNPK_TILE_KERNEL=reg (the register-staged kernel everywhere) in a subprocess gives the default route's tables."""
    host = make_fastq(np.random.default_rng(17), 4000, 0, 400, lower_frac=0.1)
    np.save(tmp_path / "chunk.npy", host)
    env = dict(os.environ, BNPK_TILE_KERNEL="reg", PYTHONPATH=ROOT)
    subprocess.run([sys.executable, "-c", _REG_SCRIPT, str(tmp_path / "chunk.npy"), str(tmp_path / "reg.npy")],
                   env=env, check=True, cwd=ROOT)
    chunk = dev(host)
    want = np.concatenate([run(ops, chunk, k, w, bins)[0] for k, w, bins in ((31, 41, 1 << 14), (15, 25, 1 << 14),
                                                                              (21, 60, 1 << 20))])
    assert np.array_equal(np.load(tmp_path / "reg.npy"), want)
    assert np.array_equal(want[: 1 << 14], chunk_oracle(host, 31, 41, 1 << 14)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("bins", [1 << 14, 1 << 24])
def test_fused_count_equals_rows_route_1m_reads(ops, bins):
    """1 M synthetic reads: the fused table equals line_split + rows_minimizer_count_canonical."""
    n = 1_000_000
    chunk = ops.synth_fastq(n)
    got, status = ops.chunk_minimizer_count_canonical(chunk, 31, 41, 3, bins)
    st = ops.read_status(status)
    assert st.n_records == n and st.n_bases == 150 * n and st.n_values == 110 * n
    starts, lens, _ = ops.line_split(chunk)
    want, _ = ops.rows_minimizer_count_canonical(chunk, starts, lens, _native.ENC_ASCII_ACGT, 31, 41, 3, bins)
    assert int(got.sum().item()) == 110 * n
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
@pytest.mark.parametrize("k,w,bins", [(21, 31, 1 << 14), (31, 41, 1 << 20), (15, 26, 1 << 14), (11, 60, 1 << 14)])
def test_fused_count_is_strand_symmetric(ops, k, w, bins):
    chunk = make_fastq(np.random.default_rng(77), 2000, 0, 300, lower_frac=0.2)
    a, _ = run(ops, chunk, k, w, bins)
    b, _ = run(ops, _revcomp_reads(chunk), k, w, bins)
    assert np.array_equal(a, b) and a.sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("k,w,bins", [(21, 31, 1 << 14), (31, 41, 1 << 14), (17, 50, 1 << 20)])
def test_status_like_plain_minimizer_count(ops, k, w, bins):
    chunk = make_fastq(np.random.default_rng(19), 3000, 0, 400, cr=True)
    chunk = chunk[:-20]                                     # an incomplete last record
    _, st = run(ops, chunk, k, w, bins)
    _, plain = ops.chunk_kmer_count(dev(chunk), k, bins, window_size=w)
    plain = ops.read_status(plain)
    assert (st.n_values, st.n_bases, st.n_complete_bytes, st.n_records) == \
        (plain.n_values, plain.n_bases, plain.n_complete_bytes, plain.n_records)


@pytest.mark.gpu
@pytest.mark.parametrize("k,w,bins", [(5, 8, 1024), (21, 31, 1 << 14), (31, 80, 1 << 20)])
def test_bad_base_like_plain(ops, k, w, bins):
    chunk = make_fastq(np.random.default_rng(3), 100, 50, 90)
    size, starts, lens = o.fastq_split(chunk)
    row, pos = 57, 13
    chunk[starts[row, 1] + pos] = ord("N")
    _, st = run(ops, chunk, k, w, bins)
    _, plain = ops.chunk_kmer_count(dev(chunk), k, bins, window_size=w)
    assert st.bad_base() == ops.read_status(plain).bad_base() == (row, pos)


@pytest.mark.gpu
def test_bad_base_raises_encoding_error_like_plain(tmp_path):
    import bionumpy_b200 as bnp
    chunk = make_fastq(np.random.default_rng(3), 100, 50, 90)
    size, starts, lens = o.fastq_split(chunk)
    chunk[starts[57, 1] + 13] = ord("N")
    p = tmp_path / "bad.fq"
    p.write_bytes(chunk.tobytes())
    errors = []
    for canonical in (False, True):
        with pytest.raises(bnp.EncodingError) as e:
            bnp.count_kmers_hashed(bnp.open(str(p)).read().sequence, 21, 1 << 14, window_size=31, canonical=canonical)
        errors.append(e.value.offset)
    assert errors[0] == errors[1] == int(lens[:57, 1].sum()) + 13


@pytest.mark.gpu
@pytest.mark.parametrize("k,w", [(1, 1), (3, 10), (15, 25), (31, 41), (21, 84)])
def test_get_minimizers_canonical_values(k, w):
    """Materialised values, including rows longer than LONG_ROW (split into pieces) and a 1-D EncodedArray."""
    import bionumpy_b200 as bnp
    from bionumpy_b200.sequence.kmers import LONG_ROW
    rng = np.random.default_rng(k + w)
    lens = np.concatenate([rng.integers(0, 200, size=300), [LONG_ROW + 5000, 2 * LONG_ROW + w]]).astype(np.int64)
    rng.shuffle(lens)
    codes = rng.integers(0, 4, size=int(lens.sum())).astype(np.uint8)
    seqs = ["".join("ACGT"[c] for c in r) for r in rows_of(codes, lens)]
    want, want_lens = canonical_minimizers(codes, lens, k, w)
    mins = bnp.get_minimizers(bnp.as_encoded_array(seqs, bnp.DNAEncoding), k, w, canonical=True)
    assert np.array_equal(mins._lens.cpu().numpy(), want_lens)
    assert np.array_equal(mins.raw().ravel().cpu().numpy(), want)
    # a 1-D EncodedArray: one row
    one = bnp.get_minimizers(bnp.as_encoded_array(seqs[int(np.argmax(lens))], bnp.DNAEncoding), k, w, canonical=True)
    i = int(np.argmax(lens))
    want_one, _ = canonical_minimizers(rows_of(codes, lens)[i], lens[i:i + 1], k, w)
    assert np.array_equal(one.raw().cpu().numpy(), want_one)


@pytest.mark.gpu
def test_minimizers_need_a_four_letter_alphabet():
    import bionumpy_b200 as bnp
    protein = bnp.as_encoded_array(["ACDEFGHIK"], bnp.AminoAcidEncoding)
    with pytest.raises(NotImplementedError):
        bnp.get_minimizers(protein, 3, 5, canonical=True).raw()


@pytest.mark.gpu
def test_saccer3_multiline_canonical_minimizers(tmp_path):
    """Every chromosome of the sacCer3 sample through the multi-line FASTA buffer: values and counts."""
    import gzip
    import torch
    import bionumpy_b200 as bnp
    raw = gzip.open(os.path.join(ROOT, "tests", "golden", "sacCer3_sample.fa.gz")).read()
    path = tmp_path / "sacCer3.fa"
    path.write_bytes(raw)
    whole = np.frombuffer((raw if raw.endswith(b"\n") else raw + b"\n") + b">", dtype=np.uint8)
    size, hs, hl, flat, seq_lens = o.multiline_fasta_split(whole)
    assert seq_lens.size == 17
    codes = o.encode_flat(flat, o.alphabet_lut("ACGT"))
    want, want_lens = canonical_minimizers(codes, seq_lens, 15, 25)
    chunk = bnp.open(str(path)).read()
    mins = bnp.get_minimizers(bnp.change_encoding(chunk.sequence, bnp.DNAEncoding), 15, 25, canonical=True)
    assert np.array_equal(mins._lens.cpu().numpy(), want_lens)
    assert np.array_equal(mins.raw().ravel().cpu().numpy(), want)
    B = 1 << 20
    hist = bnp.count_kmers_hashed(chunk.sequence, 15, B, window_size=25, canonical=True)
    assert torch.equal(hist.cpu(), torch.from_numpy(o.count_bucketed_flat(want, B)))


@pytest.mark.gpu
@pytest.mark.parametrize("k,w,bins", [(5, 9, 4 ** 5), (21, 31, 1 << 14), (31, 41, 1 << 24)])
def test_dispatcher_op_equals_ctypes(ops, k, w, bins):
    import torch
    from bionumpy_b200 import torch_ops
    tops = torch_ops.load()
    chunk = dev(make_fastq(np.random.default_rng(9), 3000, 0, 300, lower_frac=0.1))
    want, _ = ops.chunk_minimizer_count_canonical(chunk, k, w, 3, bins)
    hist = torch.zeros(bins, dtype=torch.int64, device="cuda")
    status = tops.chunk_minimizer_count_canonical(chunk, k, w, 3, hist)
    assert torch.equal(hist, want)
    assert ops.read_status(status).n_values == int(want.sum().item())


@pytest.mark.gpu
@pytest.mark.parametrize("k,w", [(5, 9), (21, 31), (31, 70)])
def test_row_ops_with_window_and_complement_xor(ops, k, w):
    """bnpk::rows_kmer_hash / rows_kmer_count with both window_size and complement_xor give canonical minimizers."""
    import torch
    from bionumpy_b200 import torch_ops
    tops = torch_ops.load()
    host = make_fastq(np.random.default_rng(11), 800, 0, 300, lower_frac=0.1)
    chunk = dev(host)
    starts, lens, _ = ops.line_split(chunk)
    size, hs, hl = o.fastq_split(host)
    codes = o.encode_flat(o.gather_rows(host, hs[:, 1], hl[:, 1]), o.alphabet_lut("ACGT"))
    want, _ = canonical_minimizers(codes, hl[:, 1], k, w)
    offsets = ops.row_offsets(lens, w - 1)
    vals, _ = tops.rows_kmer_hash(chunk, starts, lens, _native.ENC_ASCII_ACGT, None, k, w, 3, offsets,
                                  int(offsets[-1].item()))
    assert np.array_equal(vals.cpu().numpy(), want)
    hist = torch.zeros(1 << 14, dtype=torch.int64, device="cuda")
    tops.rows_kmer_count(chunk, starts, lens, _native.ENC_ASCII_ACGT, None, k, w, 3, hist)
    assert np.array_equal(hist.cpu().numpy(), o.count_bucketed_flat(want, 1 << 14))


@pytest.mark.gpu
@pytest.mark.parametrize("k,w,bins", [(21, 31, 1 << 14), (31, 41, 1 << 20), (5, 9, 4 ** 5)])
def test_file_buffer_takes_the_fused_route(ops, tmp_path, monkeypatch, k, w, bins):
    """count_kmers_hashed(..., window_size=w, canonical=True) on a bnp.open buffer runs the fused count (the rows route
    is made to fail) and gives the rows-route table; count_encoded(get_minimizers(..., canonical=True)) of the same
    sequences (get_minimizers takes DNAEncoding, so they go through change_encoding) gives it too."""
    import bionumpy_b200 as bnp
    from bionumpy_b200 import ops as ops_mod
    chunk = make_fastq(np.random.default_rng(13), 3000, 0, 300, lower_frac=0.1)
    p = tmp_path / "reads.fq"
    p.write_bytes(chunk.tobytes())
    B = bins
    seqs = bnp.open(str(p)).read().sequence
    rows_route, _ = ops.rows_minimizer_count_canonical(seqs._data, seqs._starts.contiguous(),
                                                       seqs._lens.contiguous(), _native.ENC_ASCII_ACGT, k, w, 3, B)
    want, _, _ = chunk_oracle(chunk, k, w, B)
    assert np.array_equal(rows_route.cpu().numpy(), want)

    def no_rows_route(*a, **kw):
        raise AssertionError("canonical minimizer count of a file buffer took the rows route")
    monkeypatch.setattr(ops_mod, "rows_minimizer_count_canonical", no_rows_route)
    seqs = bnp.open(str(p)).read().sequence
    got = bnp.count_kmers_hashed(seqs, k, B, window_size=w, canonical=True)
    assert np.array_equal(got.cpu().numpy(), want)
    monkeypatch.undo()
    if B == 4 ** k:
        mins = bnp.get_minimizers(bnp.change_encoding(seqs, bnp.DNAEncoding), k, w, canonical=True)
        assert np.array_equal(bnp.count_encoded(mins, axis=None).counts.cpu().numpy(), want)


@pytest.mark.gpu
def test_overflow_falls_back_to_the_rows_route(ops, tmp_path, monkeypatch):
    """A fused count that reports BNPK_ST_OVERFLOW (incomplete counts) is redone on the rows route."""
    import bionumpy_b200 as bnp
    from bionumpy_b200 import ops as ops_mod
    chunk = make_fastq(np.random.default_rng(23), 2000, 0, 300)
    p = tmp_path / "reads.fq"
    p.write_bytes(chunk.tobytes())
    fused = ops_mod.chunk_minimizer_count_canonical
    calls = []

    def overflowing(*a, **kw):
        hist, status = fused(*a, **kw)
        hist.zero_()
        status[_native.ST_OVERFLOW] = 1
        calls.append(1)
        return hist, status
    monkeypatch.setattr(ops_mod, "chunk_minimizer_count_canonical", overflowing)
    got = bnp.count_kmers_hashed(bnp.open(str(p)).read().sequence, 21, 1 << 14, window_size=31, canonical=True)
    assert calls and np.array_equal(got.cpu().numpy(), chunk_oracle(chunk, 21, 31, 1 << 14)[0])
