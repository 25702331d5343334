// torch_ops.cpp -- TORCH_LIBRARY(bnpk, ...): the k-mer hot path as PyTorch dispatcher ops.
//
// north_star: "the ragged-array and k-mer kernels bound through PyTorch's C++/CUDA extension ABI".  This file is that
// binding: a thin layer over the C-ABI of libbnpk.so (include/bnpk.h), built into libbnpk_torch.so.  Every op
//   * runs on the device of its tensors (CUDAGuard) and on torch's current stream of that device,
//   * allocates its outputs, its status block and its look-back workspace from torch's caching allocator PER CALL --
//     so two streams (or two threads) never share scratch state, and a buffer is reused only in stream order,
//   * never synchronises: the status block comes back as a tensor, the Python layer reads it when it wants to.
// It replaces the reference's `bnp.set_backend(cupy)` seam (bionumpy/__init__.py:47-94) for this path; the functions
// each op stands for are named in include/bnpk.h.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>
#include <torch/torch.h>

#include "../../include/bnpk.h"

namespace {

using torch::Tensor;

void check(int rc, const char *what) {
    TORCH_CHECK(rc == 0, "bnpk::", what, ": ", bnpk_last_error(), " (code ", rc, ")");
}
const uint8_t *u8(const Tensor &t) { return t.defined() && t.numel() ? t.data_ptr<uint8_t>() : nullptr; }
void need(const Tensor &t, c10::ScalarType st, const char *name) {
    TORCH_CHECK(t.is_cuda() && t.is_contiguous() && t.scalar_type() == st, "bnpk: ", name,
                " must be a contiguous CUDA tensor of the right dtype");
}
void *cur_stream(const Tensor &t) { return (void *)at::cuda::getCurrentCUDAStream(t.get_device()).stream(); }
Tensor new_status(const Tensor &like) {
    Tensor st = torch::empty({BNPK_ST_WORDS}, like.options().dtype(torch::kInt64));
    check(bnpk_status_init(st.data_ptr<int64_t>(), cur_stream(like)), "status_init");
    return st;
}
Tensor new_workspace(const Tensor &like, size_t n) {
    return torch::empty({(int64_t)bnpk_tile_workspace_bytes(n)}, like.options().dtype(torch::kUInt8));
}

// K6: chunk bytes -> histogram (accumulated into hist).  Returns the status block.
Tensor chunk_kmer_count(const Tensor &chunk, int64_t k, int64_t window_size, Tensor hist, int64_t lines_per_entry,
                        int64_t header_char, bool check_plus, int64_t trim_cr, int64_t enc_mode,
                        const c10::optional<Tensor> &lut, int64_t hist_mode) {
    need(chunk, torch::kUInt8, "chunk");
    need(hist, torch::kInt64, "hist");
    TORCH_CHECK(hist.get_device() == chunk.get_device(), "bnpk: chunk and hist on different devices");
    c10::cuda::CUDAGuard guard(chunk.device());
    Tensor status = new_status(chunk);
    const size_t n = (size_t)chunk.numel();
    Tensor ws = new_workspace(chunk, n);
    check(bnpk_chunk_kmer_count(chunk.data_ptr<uint8_t>(), n, 0, n, 1, (int)lines_per_entry, (uint8_t)header_char,
                                check_plus, (int)trim_cr, (int)enc_mode, lut ? u8(*lut) : nullptr, (int)k,
                                (int)window_size, hist.numel(), (int)hist_mode, hist.data_ptr<int64_t>(),
                                status.data_ptr<int64_t>(), ws.data_ptr<uint8_t>(), (size_t)ws.numel(), cur_stream(chunk)),
          "chunk_kmer_count");
    return status;
}

// K6 on canonical k-mers (min of a k-mer and its reverse complement): accumulated into hist.  Returns the status block.
Tensor chunk_kmer_count_canonical(const Tensor &chunk, int64_t k, int64_t complement_xor, Tensor hist,
                                  int64_t lines_per_entry, int64_t header_char, bool check_plus, int64_t trim_cr,
                                  int64_t enc_mode, const c10::optional<Tensor> &lut, int64_t hist_mode) {
    need(chunk, torch::kUInt8, "chunk");
    need(hist, torch::kInt64, "hist");
    TORCH_CHECK(hist.get_device() == chunk.get_device(), "bnpk: chunk and hist on different devices");
    c10::cuda::CUDAGuard guard(chunk.device());
    Tensor status = new_status(chunk);
    const size_t n = (size_t)chunk.numel();
    Tensor ws = new_workspace(chunk, n);
    check(bnpk_chunk_kmer_count_canonical(chunk.data_ptr<uint8_t>(), n, 0, n, 1, (int)lines_per_entry,
                                          (uint8_t)header_char, check_plus, (int)trim_cr, (int)enc_mode,
                                          lut ? u8(*lut) : nullptr, (int)k, (int)complement_xor, hist.numel(),
                                          (int)hist_mode, hist.data_ptr<int64_t>(), status.data_ptr<int64_t>(),
                                          ws.data_ptr<uint8_t>(), (size_t)ws.numel(), cur_stream(chunk)),
          "chunk_kmer_count_canonical");
    return status;
}

// K6 on canonical minimizers (min over each window of min(k-mer, reverse complement)): accumulated into hist.  Returns
// the status block.
Tensor chunk_minimizer_count_canonical(const Tensor &chunk, int64_t k, int64_t window_size, int64_t complement_xor,
                                       Tensor hist, int64_t lines_per_entry, int64_t header_char, bool check_plus,
                                       int64_t trim_cr, int64_t enc_mode, const c10::optional<Tensor> &lut,
                                       int64_t hist_mode) {
    need(chunk, torch::kUInt8, "chunk");
    need(hist, torch::kInt64, "hist");
    TORCH_CHECK(hist.get_device() == chunk.get_device(), "bnpk: chunk and hist on different devices");
    c10::cuda::CUDAGuard guard(chunk.device());
    Tensor status = new_status(chunk);
    const size_t n = (size_t)chunk.numel();
    Tensor ws = new_workspace(chunk, n);
    check(bnpk_chunk_minimizer_count_canonical(chunk.data_ptr<uint8_t>(), n, 0, n, 1, (int)lines_per_entry,
                                               (uint8_t)header_char, check_plus, (int)trim_cr, (int)enc_mode,
                                               lut ? u8(*lut) : nullptr, (int)k, (int)window_size, (int)complement_xor,
                                               hist.numel(), (int)hist_mode, hist.data_ptr<int64_t>(),
                                               status.data_ptr<int64_t>(), ws.data_ptr<uint8_t>(), (size_t)ws.numel(),
                                               cur_stream(chunk)),
          "chunk_minimizer_count_canonical");
    return status;
}

// K1: (starts int64[max_rows], lens int32[max_rows], status)
std::tuple<Tensor, Tensor, Tensor> line_split(const Tensor &chunk, int64_t lines_per_entry, int64_t field_line,
                                              int64_t start_offset, int64_t header_char, bool check_plus,
                                              int64_t trim_cr, int64_t max_rows) {
    need(chunk, torch::kUInt8, "chunk");
    c10::cuda::CUDAGuard guard(chunk.device());
    Tensor starts = torch::empty({max_rows}, chunk.options().dtype(torch::kInt64));
    Tensor lens = torch::empty({max_rows}, chunk.options().dtype(torch::kInt32));
    Tensor status = new_status(chunk);
    const size_t n = (size_t)chunk.numel();
    Tensor ws = new_workspace(chunk, n);
    check(bnpk_line_split(chunk.data_ptr<uint8_t>(), n, (int)lines_per_entry, (int)field_line, (int)start_offset,
                          (uint8_t)header_char, check_plus, (int)trim_cr, starts.data_ptr<int64_t>(),
                          lens.data_ptr<int32_t>(), (size_t)max_rows, status.data_ptr<int64_t>(), ws.data_ptr<uint8_t>(),
                          (size_t)ws.numel(), cur_stream(chunk)),
          "line_split");
    return {starts, lens, status};
}

Tensor row_offsets(const Tensor &lens, int64_t shrink) {
    need(lens, torch::kInt32, "lens");
    c10::cuda::CUDAGuard guard(lens.device());
    Tensor out = torch::empty({lens.numel() + 1}, lens.options().dtype(torch::kInt64));
    Tensor ws = new_workspace(lens, (size_t)std::max<int64_t>(lens.numel(), 1));
    check(bnpk_row_offsets(lens.data_ptr<int32_t>(), (size_t)lens.numel(), (int)shrink, out.data_ptr<int64_t>(),
                           ws.data_ptr<uint8_t>(), (size_t)ws.numel(), cur_stream(lens)),
          "row_offsets");
    return out;
}

void need_rows(const Tensor &base, const Tensor &starts, const Tensor &lens) {
    need(base, torch::kUInt8, "base");
    need(starts, torch::kInt64, "starts");
    need(lens, torch::kInt32, "lens");
    TORCH_CHECK(starts.numel() == lens.numel(), "bnpk: starts and lens differ in length");
}

// K2: codes uint8[total] (total = offsets[-1], given by the caller: no sync here)
std::tuple<Tensor, Tensor> rows_encode(const Tensor &base, const Tensor &starts, const Tensor &lens, int64_t enc_mode,
                                       const c10::optional<Tensor> &lut, const Tensor &offsets, int64_t total) {
    need_rows(base, starts, lens);
    c10::cuda::CUDAGuard guard(base.device());
    Tensor out = torch::empty({total}, base.options());
    Tensor status = new_status(base);
    check(bnpk_rows_encode(base.data_ptr<uint8_t>(), (size_t)base.numel(), starts.data_ptr<int64_t>(),
                           lens.data_ptr<int32_t>(), (size_t)lens.numel(), (int)enc_mode, lut ? u8(*lut) : nullptr,
                           offsets.data_ptr<int64_t>(), out.data_ptr<uint8_t>(), status.data_ptr<int64_t>(), cur_stream(base)),
          "rows_encode");
    return {out, status};
}

// K3 / K4: hashes or minimizers int64[total]
std::tuple<Tensor, Tensor> rows_kmer_hash(const Tensor &base, const Tensor &starts, const Tensor &lens, int64_t enc_mode,
                                          const c10::optional<Tensor> &lut, int64_t k, int64_t window_size,
                                          int64_t complement_xor, const Tensor &offsets, int64_t total) {
    need_rows(base, starts, lens);
    c10::cuda::CUDAGuard guard(base.device());
    Tensor out = torch::empty({total}, base.options().dtype(torch::kInt64));
    Tensor status = new_status(base);
    const uint8_t *l = lut ? u8(*lut) : nullptr;
    int rc;
    if (window_size && complement_xor)
        rc = bnpk_rows_minimizers_canonical(base.data_ptr<uint8_t>(), (size_t)base.numel(), starts.data_ptr<int64_t>(),
                                            lens.data_ptr<int32_t>(), (size_t)lens.numel(), (int)enc_mode, l, (int)k,
                                            (int)window_size, (int)complement_xor, offsets.data_ptr<int64_t>(),
                                            out.data_ptr<int64_t>(), status.data_ptr<int64_t>(), cur_stream(base));
    else if (window_size)
        rc = bnpk_rows_minimizers(base.data_ptr<uint8_t>(), (size_t)base.numel(), starts.data_ptr<int64_t>(), lens.data_ptr<int32_t>(),
                                  (size_t)lens.numel(), (int)enc_mode, l, (int)k, (int)window_size, offsets.data_ptr<int64_t>(),
                                  out.data_ptr<int64_t>(), status.data_ptr<int64_t>(), cur_stream(base));
    else if (complement_xor)
        rc = bnpk_rows_kmer_hash_canonical(base.data_ptr<uint8_t>(), (size_t)base.numel(), starts.data_ptr<int64_t>(),
                                           lens.data_ptr<int32_t>(), (size_t)lens.numel(), (int)enc_mode, l, (int)k,
                                           (int)complement_xor, offsets.data_ptr<int64_t>(), out.data_ptr<int64_t>(),
                                           status.data_ptr<int64_t>(), cur_stream(base));
    else
        rc = bnpk_rows_kmer_hash(base.data_ptr<uint8_t>(), (size_t)base.numel(), starts.data_ptr<int64_t>(), lens.data_ptr<int32_t>(),
                                 (size_t)lens.numel(), (int)enc_mode, l, (int)k, offsets.data_ptr<int64_t>(),
                                 out.data_ptr<int64_t>(), status.data_ptr<int64_t>(), cur_stream(base));
    check(rc, "rows_kmer_hash");
    return {out, status};
}

// K3/K4 + K5 on a ragged view (accumulates into hist)
Tensor rows_kmer_count(const Tensor &base, const Tensor &starts, const Tensor &lens, int64_t enc_mode,
                       const c10::optional<Tensor> &lut, int64_t k, int64_t window_size, int64_t complement_xor,
                       Tensor hist, int64_t hist_mode) {
    need_rows(base, starts, lens);
    need(hist, torch::kInt64, "hist");
    c10::cuda::CUDAGuard guard(base.device());
    Tensor status = new_status(base);
    const uint8_t *l = lut ? u8(*lut) : nullptr;
    int rc;
    if (window_size && complement_xor)
        rc = bnpk_rows_minimizer_count_canonical(base.data_ptr<uint8_t>(), (size_t)base.numel(), starts.data_ptr<int64_t>(),
                                                 lens.data_ptr<int32_t>(), (size_t)lens.numel(), (int)enc_mode, l, (int)k,
                                                 (int)window_size, (int)complement_xor, hist.numel(), (int)hist_mode,
                                                 hist.data_ptr<int64_t>(), status.data_ptr<int64_t>(), cur_stream(base));
    else if (complement_xor)
        rc = bnpk_rows_kmer_count_canonical(base.data_ptr<uint8_t>(), (size_t)base.numel(), starts.data_ptr<int64_t>(),
                                            lens.data_ptr<int32_t>(), (size_t)lens.numel(), (int)enc_mode, l, (int)k,
                                            (int)complement_xor, hist.numel(), (int)hist_mode, hist.data_ptr<int64_t>(),
                                            status.data_ptr<int64_t>(), cur_stream(base));
    else
        rc = bnpk_rows_kmer_count(base.data_ptr<uint8_t>(), (size_t)base.numel(), starts.data_ptr<int64_t>(), lens.data_ptr<int32_t>(),
                                  (size_t)lens.numel(), (int)enc_mode, l, (int)k, (int)window_size, hist.numel(), (int)hist_mode,
                                  hist.data_ptr<int64_t>(), status.data_ptr<int64_t>(), cur_stream(base));
    check(rc, "rows_kmer_count");
    return status;
}

Tensor rows_reverse_complement(const Tensor &base, const Tensor &starts, const Tensor &lens, const Tensor &lut,
                               const Tensor &offsets, int64_t total) {
    need_rows(base, starts, lens);
    need(lut, torch::kUInt8, "lut");
    c10::cuda::CUDAGuard guard(base.device());
    Tensor out = torch::empty({total}, base.options());
    check(bnpk_rows_reverse_complement(base.data_ptr<uint8_t>(), (size_t)base.numel(), starts.data_ptr<int64_t>(),
                                       lens.data_ptr<int32_t>(), (size_t)lens.numel(), lut.data_ptr<uint8_t>(),
                                       offsets.data_ptr<int64_t>(), out.data_ptr<uint8_t>(), cur_stream(base)),
          "rows_reverse_complement");
    return out;
}

// K5 (accumulates into hist)
Tensor bincount(const Tensor &values, Tensor hist, int64_t hist_mode) {
    need(values, torch::kInt64, "values");
    need(hist, torch::kInt64, "hist");
    c10::cuda::CUDAGuard guard(values.device());
    Tensor status = new_status(values);
    check(bnpk_bincount(values.data_ptr<int64_t>(), (size_t)values.numel(), hist.numel(), (int)hist_mode,
                        hist.data_ptr<int64_t>(), status.data_ptr<int64_t>(), cur_stream(values)),
          "bincount");
    return status;
}

}  // namespace

TORCH_LIBRARY(bnpk, m) {
    m.def("chunk_kmer_count(Tensor chunk, int k, int window_size, Tensor(a!) hist, int lines_per_entry=4, "
          "int header_char=64, bool check_plus=True, int trim_cr=-1, int enc_mode=0, Tensor? lut=None, "
          "int hist_mode=0) -> Tensor");
    m.def("chunk_kmer_count_canonical(Tensor chunk, int k, int complement_xor, Tensor(a!) hist, int lines_per_entry=4, "
          "int header_char=64, bool check_plus=True, int trim_cr=-1, int enc_mode=0, Tensor? lut=None, "
          "int hist_mode=0) -> Tensor");
    m.def("chunk_minimizer_count_canonical(Tensor chunk, int k, int window_size, int complement_xor, Tensor(a!) hist, "
          "int lines_per_entry=4, int header_char=64, bool check_plus=True, int trim_cr=-1, int enc_mode=0, "
          "Tensor? lut=None, int hist_mode=0) -> Tensor");
    m.def("line_split(Tensor chunk, int lines_per_entry, int field_line, int start_offset, int header_char, "
          "bool check_plus, int trim_cr, int max_rows) -> (Tensor, Tensor, Tensor)");
    m.def("row_offsets(Tensor lens, int shrink) -> Tensor");
    m.def("rows_encode(Tensor base, Tensor starts, Tensor lens, int enc_mode, Tensor? lut, Tensor offsets, int total) "
          "-> (Tensor, Tensor)");
    m.def("rows_kmer_hash(Tensor base, Tensor starts, Tensor lens, int enc_mode, Tensor? lut, int k, int window_size, "
          "int complement_xor, Tensor offsets, int total) -> (Tensor, Tensor)");
    m.def("rows_kmer_count(Tensor base, Tensor starts, Tensor lens, int enc_mode, Tensor? lut, int k, int window_size, "
          "int complement_xor, Tensor(a!) hist, int hist_mode=0) -> Tensor");
    m.def("rows_reverse_complement(Tensor base, Tensor starts, Tensor lens, Tensor lut, Tensor offsets, int total) -> Tensor");
    m.def("bincount(Tensor values, Tensor(a!) hist, int hist_mode=0) -> Tensor");
}

TORCH_LIBRARY_IMPL(bnpk, CUDA, m) {
    m.impl("chunk_kmer_count", &chunk_kmer_count);
    m.impl("chunk_kmer_count_canonical", &chunk_kmer_count_canonical);
    m.impl("chunk_minimizer_count_canonical", &chunk_minimizer_count_canonical);
    m.impl("line_split", &line_split);
    m.impl("row_offsets", &row_offsets);
    m.impl("rows_encode", &rows_encode);
    m.impl("rows_kmer_hash", &rows_kmer_hash);
    m.impl("rows_kmer_count", &rows_kmer_count);
    m.impl("rows_reverse_complement", &rows_reverse_complement);
    m.impl("bincount", &bincount);
}
