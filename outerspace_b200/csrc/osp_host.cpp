// osp_host.cpp -- host side of the drop-in surface: the .mtx loader and COO->CSR/CSC builders.
//
// north_star keeps "the same .mtx loaders, the same CSR/CSC operand structs": these are the
// C-ABI forms of readcoo (simulator/SimSpGEMM.cpp:55-100) and coo2csr<transpose> + dupcheck
// (SimSpGEMM.cpp:43-53,102-152).  They are host code in the reference and stay available as host code here; the line
// grammar is shared with the device parser of osp_readcoo_device (osp_mtx_grammar.h, osp_mtx.cuh).
//
// Behaviour kept: blank and '%' lines are skipped; the first remaining line is "NRow NCol NNZ";
// entries are 1-based; a missing value means 1.0; values are parsed as double then narrowed to
// float; `symmetric` mirrors off-diagonal entries; duplicates make coo2csr fail with 233.
// Deliberate divergences (DESIGN.md "Divergences"): an index >= N is reported as OSP_ERR_INDEX
// instead of writing out of bounds, and the reference's trailing fix-up corner that turns every
// pos into nnz when all non-zeros share one slice (SimSpGEMM.cpp:143-148) is not reproduced.
#include "osp_mtx_host.h"
#include "osp_mtx_grammar.h"

#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <string>
#include <thread>
#include <vector>

namespace {

// Parses an unsigned decimal field the way sscanf("%zu") does: skips white space, accepts digits.
bool parse_u64(const char *&s, uint64_t &out) {
    while (*s == ' ' || *s == '\t' || *s == '\r' || *s == '\n' || *s == '\v' || *s == '\f') s++;
    char *end = nullptr;
    errno = 0;
    unsigned long long v = std::strtoull(s, &end, 10);
    if (end == s) return false;
    out = v;
    s = end;
    return true;
}
bool parse_f64(const char *&s, double &out) {
    char *end = nullptr;
    double v = std::strtod(s, &end);
    if (end == s) return false;
    out = v;
    s = end;
    return true;
}

#pragma pack(push, 1)
struct HostElem {
    uint32_t idx;
    float val;
};
#pragma pack(pop)

}  // namespace


// Parses Matrix-Market text held in memory (the reference reads from a std::istream, SimSpGEMM.cpp:55).
//
// The reference's loader is one getline + sscanf("%zu %zu %lf") per line on one thread (SimSpGEMM.cpp:60-97); at
// config 4's size (6.7e7 entries, 1.3 GB of text) that is the longest step of an end-to-end run (SURVEY 8f rank 2).
// Here the header is found serially, then the body is cut at line boundaries into one piece per host thread.  A line of
// the plain shape  <digits> <digits> [<decimal number>]  is parsed in place: the value by Clinger's exact fast path (at
// most 15 significant digits and |decimal exponent| <= 22: mantissa and power of ten are both exact doubles, so one
// multiply or divide rounds correctly -- the same double strtod / "%lf" produce, then the same narrowing to float).
// Every other line (signs on the indices, inf/nan, hex floats, long mantissas, ...) goes through the strtoull / strtod
// path on a NUL-terminated copy, so the result is identical in every case; entry order is the file's.
namespace osp_mtx {

bool header_line(const std::string &line, uint64_t hdr[3]) {
    size_t first = line.find_first_not_of(" \t\r");
    if (first == std::string::npos || line[first] == '%') return false;
    const char *s = line.c_str();
    if (parse_u64(s, hdr[0]) && parse_u64(s, hdr[1])) parse_u64(s, hdr[2]);
    return true;
}

// (NUL-terminated copy)
int slow_line(const std::string &line, int symmetric, Piece &out) {
    const char *s = line.c_str();
    uint64_t r = 0, col = 0;
    double v = 1.0;
    if (!parse_u64(s, r) || !parse_u64(s, col)) return OSP_ERR_INVALID;   // the reference reads garbage here; we refuse
    double parsed;
    if (parse_f64(s, parsed)) v = parsed;
    out.rows.push_back(uint32_t(r - 1)); out.cols.push_back(uint32_t(col - 1)); out.vals.push_back(float(v));
    if (symmetric && r != col) {
        out.rows.push_back(uint32_t(col - 1)); out.cols.push_back(uint32_t(r - 1)); out.vals.push_back(float(v));
    }
    return OSP_OK;
}

}  // namespace osp_mtx

namespace {

using osp_mtx::Piece;

void parse_piece(const char *p, const char *end, int symmetric, Piece &out) {
    std::string copy;
    while (p < end) {
        const char *nl = static_cast<const char *>(std::memchr(p, '\n', size_t(end - p)));
        const char *le = nl ? nl : end;
        const char *q = p;
        p = nl ? nl + 1 : end;
        uint64_t r = 0, col = 0;
        double v = 1.0;
        const int kind = osp_mtx::plain_line(q, le, r, col, v);
        if (kind == osp_mtx::LINE_SKIP) continue;
        if (kind == osp_mtx::LINE_SLOW) {
            copy.assign(q, size_t(le - q));
            if (int rc = osp_mtx::slow_line(copy, symmetric, out)) { out.err = rc; return; }
            continue;
        }
        out.rows.push_back(uint32_t(r - 1)); out.cols.push_back(uint32_t(col - 1)); out.vals.push_back(float(v));
        if (symmetric && r != col) {
            out.rows.push_back(uint32_t(col - 1)); out.cols.push_back(uint32_t(r - 1)); out.vals.push_back(float(v));
        }
    }
}

unsigned host_threads(uint64_t bytes) {
    if (const char *env = std::getenv("OSP_HOST_THREADS")) {              // explicit: exactly that many (tests)
        const unsigned n = unsigned(std::strtoul(env, nullptr, 10));
        return unsigned(std::min<uint64_t>(std::max(1u, std::min(n, 64u)), bytes / 64 + 1));
    }
    const unsigned n = std::max(1u, std::min(std::thread::hardware_concurrency(), 64u));
    return unsigned(std::min<uint64_t>(n, bytes / (1u << 20) + 1));      // at least 1 MB of text per thread
}

}  // namespace

// No C++ exception crosses the C ABI: allocation failures become OSP_ERR_OOM, anything else OSP_ERR_INVALID.
#define OSP_NOTHROW(expr)                                   \
    try { return (expr); }                                  \
    catch (const std::bad_alloc &) { return OSP_ERR_OOM; }  \
    catch (...) { return OSP_ERR_INVALID; }

extern "C" {

static int osp_readcoo_buffer_impl(const char *text, uint64_t len, int symmetric, osp_coo **out) {
    if ((!text && len) || !out) return OSP_ERR_INVALID;
    *out = nullptr;
    // ---- header: the first line that is neither blank nor a comment (SimSpGEMM.cpp:66-88) ----
    uint64_t at = 0;
    uint64_t hdr[3] = {0, 0, 0};
    bool header_seen = false;
    while (at < len && !header_seen) {
        uint64_t nl = at;
        while (nl < len && text[nl] != '\n') nl++;
        const std::string line(text + at, nl - at);
        at = std::min<uint64_t>(nl + 1, len);
        header_seen = osp_mtx::header_line(line, hdr);
    }
    osp_coo *c = new osp_coo();
    c->nrow = hdr[0]; c->ncol = hdr[1]; c->nnz_header = hdr[2];
    // ---- body: one piece per thread, cut at line boundaries ----
    const char *body = text + at, *end = text + len;
    const unsigned T = host_threads(uint64_t(end - body));
    std::vector<const char *> cut(T + 1, end);
    cut[0] = body;
    for (unsigned i = 1; i < T; i++) {
        const char *g = body + (uint64_t(end - body) * i) / T;
        if (g < cut[i - 1]) g = cut[i - 1];
        const char *nl = static_cast<const char *>(std::memchr(g, '\n', size_t(end - g)));
        cut[i] = nl ? nl + 1 : end;
    }
    std::vector<Piece> pieces(T);
    const size_t guess = size_t((symmetric ? 2 : 1) * hdr[2] / T + 16);
    auto work = [&](unsigned i) {
        try {            // (an exception must not leave a worker thread: std::terminate)
            // the header's NNZ is untrusted: an entry takes at least four bytes of text ("1 1\n")
            const size_t cap = std::min(guess, size_t((symmetric ? 2 : 1) * uint64_t(cut[i + 1] - cut[i]) / 4 + 16));
            if (hdr[2] < (1ull << 32)) { pieces[i].rows.reserve(cap); pieces[i].cols.reserve(cap); pieces[i].vals.reserve(cap); }
            parse_piece(cut[i], cut[i + 1], symmetric, pieces[i]);
        } catch (const std::bad_alloc &) {
            pieces[i].err = OSP_ERR_OOM;
        } catch (...) {
            pieces[i].err = OSP_ERR_INVALID;
        }
    };
    if (T == 1) {
        work(0);
    } else {
        std::vector<std::thread> th;
        for (unsigned i = 1; i < T; i++) th.emplace_back(work, i);
        work(0);
        for (auto &t : th) t.join();
    }
    for (const Piece &pc : pieces)
        if (pc.err) { delete c; return pc.err; }
    // ---- concatenate in file order ----
    std::vector<size_t> off(T + 1, 0);
    for (unsigned i = 0; i < T; i++) off[i + 1] = off[i] + pieces[i].rows.size();
    c->rows.resize(off[T]); c->cols.resize(off[T]); c->vals.resize(off[T]);
    auto gather = [&](unsigned i) {
        const size_t n = pieces[i].rows.size();
        if (!n) return;
        std::memcpy(c->rows.data() + off[i], pieces[i].rows.data(), n * 4);
        std::memcpy(c->cols.data() + off[i], pieces[i].cols.data(), n * 4);
        std::memcpy(c->vals.data() + off[i], pieces[i].vals.data(), n * 4);
        Piece().rows.swap(pieces[i].rows); Piece().cols.swap(pieces[i].cols); Piece().vals.swap(pieces[i].vals);
    };
    if (T == 1) {
        c->rows.swap(pieces[0].rows); c->cols.swap(pieces[0].cols); c->vals.swap(pieces[0].vals);
    } else {
        std::vector<std::thread> th;
        for (unsigned i = 1; i < T; i++) th.emplace_back(gather, i);
        gather(0);
        for (auto &t : th) t.join();
    }
    *out = c;
    return OSP_OK;
}

static int osp_readcoo_impl(const char *path, int symmetric, osp_coo **out) {
    if (!path || !out) return OSP_ERR_INVALID;
    *out = nullptr;
    FILE *f = std::fopen(path, "rb");
    if (!f) return OSP_ERR_IO;
    std::string text;
    if (std::fseek(f, 0, SEEK_END) == 0) {
        const long sz = std::ftell(f);
        if (sz > 0) text.reserve(size_t(sz));
        std::rewind(f);
    }
    std::vector<char> buf(1 << 22);
    size_t n;
    while ((n = std::fread(buf.data(), 1, buf.size(), f)) > 0) text.append(buf.data(), n);
    std::fclose(f);
    return osp_readcoo_buffer(text.data(), text.size(), symmetric, out);
}

int osp_coo_dims(const osp_coo *c, uint64_t *nrow, uint64_t *ncol, uint64_t *nnz) {
    if (!c) return OSP_ERR_INVALID;
    if (nrow) *nrow = c->nrow;
    if (ncol) *ncol = c->ncol;
    if (nnz) *nnz = c->ctx ? c->d_nnz : c->rows.size();
    return OSP_OK;
}

static int osp_coo_copy_impl(const osp_coo *c, uint32_t *rows, uint32_t *cols, float *vals) {
    if (!c) return OSP_ERR_INVALID;
    if (c->ctx) return osp_coo_device_copy(c, rows, cols, vals);
    size_t n = c->rows.size();
    if (n && (!rows || !cols || !vals)) return OSP_ERR_INVALID;
    if (n) {
        std::memcpy(rows, c->rows.data(), n * 4);
        std::memcpy(cols, c->cols.data(), n * 4);
        std::memcpy(vals, c->vals.data(), n * 4);
    }
    return OSP_OK;
}

void osp_coo_free(osp_coo *c) {
    if (c && c->ctx) osp_coo_device_free(c);
    delete c;
}

// Stable counting passes instead of the reference's comparison sort (std::sort by (row, col) or (col, row),
// SimSpGEMM.cpp:113-120): the resulting order (major, minor) is the same because keys are unique or the call fails.
// The order the triplets arrive in decides how many passes are needed -- a .mtx written from a compressed matrix
// (scipy.io.mmwrite of a csr_matrix, NN_models/util.py:61-62) is already sorted by (row, col):
//   sorted by (major, minor): no pass, the elements are copied in place            (CSR from a row-major file)
//   sorted by (minor, major): one stable pass by major                             (CSC from a row-major file)
//   anything else:            stable pass by minor, then stable pass by major
static int osp_coo2csr_impl(uint64_t nnz, const uint32_t *rows, const uint32_t *cols, const float *vals, uint64_t N, int transpose,
                uint64_t *pos, void *data) {
    if (!pos || (nnz && (!rows || !cols || !vals || !data))) return OSP_ERR_INVALID;
    const uint32_t *major = transpose ? cols : rows;
    const uint32_t *minor = transpose ? rows : cols;
    uint64_t minor_range = 0;
    bool by_major_minor = true, by_minor_major = true;       // non-descending in that lexicographic order
    for (uint64_t i = 0; i < nnz; i++) {
        if (major[i] >= N) return OSP_ERR_INDEX;
        if (uint64_t(minor[i]) + 1 > minor_range) minor_range = uint64_t(minor[i]) + 1;
        if (i) {
            if (major[i] < major[i - 1] || (major[i] == major[i - 1] && minor[i] < minor[i - 1])) by_major_minor = false;
            if (minor[i] < minor[i - 1] || (minor[i] == minor[i - 1] && major[i] < major[i - 1])) by_minor_major = false;
        }
    }
    for (uint64_t i = 0; i <= N; i++) pos[i] = 0;
    for (uint64_t i = 0; i < nnz; i++) pos[major[i] + 1]++;
    for (uint64_t i = 0; i < N; i++) pos[i + 1] += pos[i];
    HostElem *out = static_cast<HostElem *>(data);
    if (by_major_minor) {
        for (uint64_t i = 0; i < nnz; i++) out[i] = HostElem{minor[i], vals[i]};
    } else {
        std::vector<uint64_t> cursor(pos, pos + N);
        if (by_minor_major) {
            for (uint64_t i = 0; i < nnz; i++) out[cursor[major[i]]++] = HostElem{minor[i], vals[i]};
        } else {
            // pass 1: order by minor; pass 2: stable order by major.  Pass 1 counts over the minor range when that is
            // not much larger than the input; ids up to 2^32 - 1 would need a 32 GB count array, so a wide range takes
            // a stable comparison sort instead (the same order)
            std::vector<uint64_t> by_minor(nnz);
            if (minor_range <= 4 * nnz + (1u << 20)) {
                std::vector<uint64_t> start(minor_range + 1, 0);
                for (uint64_t i = 0; i < nnz; i++) start[minor[i] + 1]++;
                for (uint64_t i = 0; i < minor_range; i++) start[i + 1] += start[i];
                for (uint64_t i = 0; i < nnz; i++) by_minor[start[minor[i]]++] = i;
            } else {
                for (uint64_t i = 0; i < nnz; i++) by_minor[i] = i;
                std::stable_sort(by_minor.begin(), by_minor.end(), [&](uint64_t x, uint64_t y) { return minor[x] < minor[y]; });
            }
            for (uint64_t j = 0; j < nnz; j++) {
                const uint64_t i = by_minor[j];
                out[cursor[major[i]]++] = HostElem{minor[i], vals[i]};
            }
        }
    }
    // dupcheck (SimSpGEMM.cpp:43-53): equal neighbours inside a slice
    for (uint64_t s = 0; s < N; s++)
        for (uint64_t e = pos[s] + 1; e < pos[s + 1]; e++)
            if (out[e].idx == out[e - 1].idx) return OSP_ERR_DUPLICATE;
    return OSP_OK;
}

// ---- compact COO (CompactCOOMatrix, common.h:52-56) -------------------------------------------------------------
// csr2compact (SimSpGEMM.cpp:154-219): group j holds the (j+1)-th non-zero of every slice that has one, slices in
// ascending order; n_groups = the longest slice.  The reference counts the slices per length, suffix-sums the counts
// and walks the slices with one cursor per group; here the suffix sum is the same and the scatter walks the slices in
// ascending order with one cursor per group as well (fill[j]++): element j of slice i lands at group_pos[j] + (slices
// before i that hold more than j non-zeros).
// A matrix without any non-zero gives zero groups (the reference indexes statNNZR[-1] there: undefined behaviour).
static int osp_csr2compact_impl(uint64_t n_major, const uint64_t *pos, const void *data, uint64_t *n_groups, uint64_t *group_pos,
                    uint32_t *rows, uint32_t *cols, float *vals) {
    if (!n_groups || (n_major && !pos)) return OSP_ERR_INVALID;
    uint64_t longest = 0;
    for (uint64_t i = 0; i < n_major; i++) {
        if (pos[i + 1] < pos[i]) return OSP_ERR_INVALID;
        longest = std::max(longest, pos[i + 1] - pos[i]);
    }
    *n_groups = longest;
    if (!group_pos) return OSP_OK;                        // size query
    const uint64_t nnz = n_major ? pos[n_major] - pos[0] : 0;
    if (nnz && (!data || !rows || !cols || !vals)) return OSP_ERR_INVALID;
    // at_least[j] = slices with more than j non-zeros (SimSpGEMM.cpp:172-185)
    std::vector<uint64_t> at_least(longest + 1, 0);
    for (uint64_t i = 0; i < n_major; i++) {
        const uint64_t len = pos[i + 1] - pos[i];
        if (len) at_least[len - 1]++;
    }
    for (uint64_t j = longest; j-- > 1;) at_least[j - 1] += at_least[j];
    group_pos[0] = 0;
    for (uint64_t j = 0; j < longest; j++) group_pos[j + 1] = group_pos[j] + at_least[j];
    const HostElem *in = static_cast<const HostElem *>(data);
    std::vector<uint64_t> fill(group_pos, group_pos + longest);          // next free place of every group
    for (uint64_t i = 0; i < n_major; i++) {
        const HostElem *e = in + pos[i];
        const uint64_t len = pos[i + 1] - pos[i];
        for (uint64_t j = 0; j < len; j++) {
            const uint64_t o = fill[j]++;
            rows[o] = uint32_t(i); cols[o] = e[j].idx; vals[o] = e[j].val;
        }
    }
    return OSP_OK;
}

// csc2rawcompact (SimSpGEMM.cpp:221-243): the COO view of a compressed matrix, one group per slice (group_pos = pos):
// row = the element's index, col = the slice id.
static int osp_csc2rawcompact_impl(uint64_t n_major, const uint64_t *pos, const void *data, uint32_t *rows, uint32_t *cols, float *vals) {
    if (n_major && !pos) return OSP_ERR_INVALID;
    const uint64_t nnz = n_major ? pos[n_major] - pos[0] : 0;
    if (nnz && (!data || !rows || !cols || !vals)) return OSP_ERR_INVALID;
    const HostElem *in = static_cast<const HostElem *>(data);
    for (uint64_t s = 0; s < n_major; s++)
        for (uint64_t e = pos[s]; e < pos[s + 1]; e++) {
            rows[e - pos[0]] = in[e].idx; cols[e - pos[0]] = uint32_t(s); vals[e - pos[0]] = in[e].val;
        }
    return OSP_OK;
}

int osp_readcoo_buffer(const char *text, uint64_t len, int symmetric, osp_coo **out) {
    OSP_NOTHROW(osp_readcoo_buffer_impl(text, len, symmetric, out));
}
int osp_readcoo(const char *path, int symmetric, osp_coo **out) {
    OSP_NOTHROW(osp_readcoo_impl(path, symmetric, out));
}
int osp_coo_copy(const osp_coo *c, uint32_t *rows, uint32_t *cols, float *vals) {
    OSP_NOTHROW(osp_coo_copy_impl(c, rows, cols, vals));
}
int osp_coo2csr(uint64_t nnz, const uint32_t *rows, const uint32_t *cols, const float *vals, uint64_t N, int transpose,
                uint64_t *pos, void *data) {
    OSP_NOTHROW(osp_coo2csr_impl(nnz, rows, cols, vals, N, transpose, pos, data));
}
int osp_csr2compact(uint64_t n_major, const uint64_t *pos, const void *data, uint64_t *n_groups, uint64_t *group_pos,
                    uint32_t *rows, uint32_t *cols, float *vals) {
    OSP_NOTHROW(osp_csr2compact_impl(n_major, pos, data, n_groups, group_pos, rows, cols, vals));
}
int osp_csc2rawcompact(uint64_t n_major, const uint64_t *pos, const void *data, uint32_t *rows, uint32_t *cols, float *vals) {
    OSP_NOTHROW(osp_csc2rawcompact_impl(n_major, pos, data, rows, cols, vals));
}
}  // extern "C"
