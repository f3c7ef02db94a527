// osp_b200.hpp -- C++ host shim over the C ABI (osp_b200.h): the reference's own names for the
// functional SpGEMM path, so that simulator/SimSpGEMM.cpp's main() (lines 841-894) can call the GPU
// engine by changing one namespace.  Header-only; link with -losp_b200.
//
//   reference (simulator/)                               this header (namespace osp_b200)
//   common.h:7-16    index_t, value_t, CSRElement        same layout (packed 8 bytes)
//   common.h:18-33   COOElement, operator<                same
//   common.h:39-49   CSRMatrix{pos,data,NRow()}, COOMatrix same
//   SimSpGEMM.cpp:55   readcoo(istream&, NRow, NCol, sym) same signature
//   SimSpGEMM.cpp:102  coo2csr<transpose>(coo, N)         same signature; throws int 233 on duplicates (:49)
//   SimOuterSPACE.cpp:44-144 TaskProvider(lmatCSC, rmatCSR) same constructor; runs multiply + merge on the GPU;
//                      getMultiplyTasks()/getMergeTasks() give the task SIZES the timing models read (:176-196);
//                      mergedResult is public and holds the intended (cscMulcsr + deduplicateCOO) result
//   SimSpGEMM.cpp:884-891 mulflops_ref                    mulflops(csc, csr)
//   common.h:52-56   CompactCOOMatrix{pos,data}           same
//   SimSpGEMM.cpp:154  csr2compact(csr)                   same signature
//   SimSpGEMM.cpp:221  csc2rawcompact(csc)                same signature
//   SimSpGEMM.cpp:247  compactMulcsr(compact, csr)        Engine::compactMulcsr: the MERGED product (the reference returns
//                                                         the unmerged partial products of every group)
//
// Errors: the reference asserts (abort) on a k-dimension mismatch and throws the int 233 on duplicate
// entries.  Here coo2csr throws 233 as well (so existing catch sites keep working); everything else
// throws osp_b200::Error carrying the C status code.
#ifndef OSP_B200_HPP
#define OSP_B200_HPP

#include <cstddef>
#include <cstdint>
#include <istream>
#include <iterator>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "osp_b200.h"

namespace osp_b200 {

typedef uint32_t index_t;
typedef float value_t;

#pragma pack(push, 1)
struct CSRElement {
    index_t idx;
    value_t val;
};
#pragma pack(pop)
static_assert(sizeof(CSRElement) == 8, "packed as in common.h:10-16");

struct COOElement {
    index_t row, col;
    value_t val;
    bool operator<(const COOElement &o) const { return row != o.row ? row < o.row : col < o.col; }
};

struct CSRMatrix {
    std::vector<size_t> pos;
    std::vector<CSRElement> data;
    size_t NRow() const { return pos.empty() ? 0 : pos.size() - 1; }
};
typedef std::vector<COOElement> COOMatrix;
static_assert(sizeof(size_t) == sizeof(uint64_t), "CSRMatrix::pos is handed to the C ABI as uint64_t[]");

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &what) : std::runtime_error(what), code(c) {}
};

inline void check(int rc, osp_ctx *ctx, const char *where) {
    if (rc != OSP_OK) throw Error(rc, std::string(where) + ": " + osp_last_error(ctx));
}

// ---- loaders (host code in the reference, host code here) ------------------------------------------
inline COOMatrix readcoo(std::istream &in, size_t &NRow, size_t &NCol, bool sym) {
    std::string text((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
    osp_coo *h = nullptr;
    check(osp_readcoo_buffer(text.data(), text.size(), sym ? 1 : 0, &h), nullptr, "readcoo");
    uint64_t nr = 0, nc = 0, nnz = 0;
    osp_coo_dims(h, &nr, &nc, &nnz);
    std::vector<uint32_t> r(nnz), c(nnz);
    std::vector<float> v(nnz);
    osp_coo_copy(h, r.data(), c.data(), v.data());
    osp_coo_free(h);
    NRow = nr; NCol = nc;
    COOMatrix coo(nnz);
    for (size_t i = 0; i < nnz; i++) coo[i] = COOElement{r[i], c[i], v[i]};
    return coo;
}

template <bool transpose = false>
CSRMatrix coo2csr(COOMatrix coo, size_t N) {
    std::vector<uint32_t> r(coo.size()), c(coo.size());
    std::vector<float> v(coo.size());
    for (size_t i = 0; i < coo.size(); i++) { r[i] = coo[i].row; c[i] = coo[i].col; v[i] = coo[i].val; }
    CSRMatrix out;
    out.pos.assign(N + 1, 0);
    out.data.resize(coo.size());
    int rc = osp_coo2csr(coo.size(), r.data(), c.data(), v.data(), N, transpose ? 1 : 0,
                         reinterpret_cast<uint64_t *>(out.pos.data()), out.data.data());
    if (rc == OSP_ERR_DUPLICATE) throw(233);            // what dupcheck throws, SimSpGEMM.cpp:49
    check(rc, nullptr, "coo2csr");
    return out;
}

struct CompactCOOMatrix {
    std::vector<size_t> pos;
    std::vector<COOElement> data;
};

inline CompactCOOMatrix from_triplets(std::vector<size_t> pos, const std::vector<uint32_t> &r, const std::vector<uint32_t> &c,
                                      const std::vector<float> &v) {
    CompactCOOMatrix out;
    out.pos = std::move(pos);
    out.data.resize(r.size());
    for (size_t i = 0; i < r.size(); i++) out.data[i] = COOElement{r[i], c[i], v[i]};
    return out;
}

inline CompactCOOMatrix csr2compact(const CSRMatrix &csr) {
    if (csr.pos.empty()) return CompactCOOMatrix();
    uint64_t groups = 0;
    const uint64_t *pos = reinterpret_cast<const uint64_t *>(csr.pos.data());
    check(osp_csr2compact(csr.NRow(), pos, csr.data.data(), &groups, nullptr, nullptr, nullptr, nullptr), nullptr, "csr2compact");
    std::vector<size_t> gpos(groups + 1, 0);
    std::vector<uint32_t> r(csr.data.size()), c(csr.data.size());
    std::vector<float> v(csr.data.size());
    check(osp_csr2compact(csr.NRow(), pos, csr.data.data(), &groups, reinterpret_cast<uint64_t *>(gpos.data()), r.data(), c.data(), v.data()),
          nullptr, "csr2compact");
    return from_triplets(std::move(gpos), r, c, v);
}

inline CompactCOOMatrix csc2rawcompact(const CSRMatrix &csc) {
    std::vector<uint32_t> r(csc.data.size()), c(csc.data.size());
    std::vector<float> v(csc.data.size());
    check(osp_csc2rawcompact(csc.NRow(), reinterpret_cast<const uint64_t *>(csc.pos.data()), csc.data.data(), r.data(), c.data(), v.data()),
          nullptr, "csc2rawcompact");
    return from_triplets(csc.pos, r, c, v);
}

inline size_t mulflops(const CSRMatrix &csc, const CSRMatrix &csr) {
    size_t f = 0;
    for (size_t i = 0; i + 1 < csr.pos.size() && i + 1 < csc.pos.size(); i++)
        f += (csc.pos[i + 1] - csc.pos[i]) * (csr.pos[i + 1] - csr.pos[i]);
    return f;
}

// ---- the engine ------------------------------------------------------------------------------------
// Triplets of a .mtx file parsed on the device (Engine::readcoo_device), resident in HBM until destroyed; destroy it
// before its Engine.
class DeviceCOO {
public:
    DeviceCOO(osp_ctx *ctx, osp_coo *h) : ctx_(ctx), h_(h) {}
    DeviceCOO(DeviceCOO &&o) noexcept : ctx_(o.ctx_), h_(o.h_) { o.h_ = nullptr; }
    DeviceCOO(const DeviceCOO &) = delete;
    DeviceCOO &operator=(const DeviceCOO &) = delete;
    ~DeviceCOO() { osp_coo_free(h_); }
    size_t size() const { uint64_t n = 0; osp_coo_dims(h_, nullptr, nullptr, &n); return n; }
    osp_coo *handle() const { return h_; }

    // coo2csr<transpose>(coo, N) + dupcheck, built on the device (throws 233 on a duplicate like coo2csr)
    template <bool transpose = false>
    CSRMatrix coo2csr(size_t N) const {
        osp_result *res = nullptr;
        int rc = osp_coo2csr_result(ctx_, h_, N, transpose ? 1 : 0, &res);
        if (rc == OSP_ERR_DUPLICATE) throw(233);
        check(rc, ctx_, "coo2csr (device)");
        CSRMatrix out;
        uint64_t rows = 0, nnz = 0;
        osp_result_dims(res, &rows, &nnz);
        out.pos.resize(rows + 1);
        out.data.resize(nnz);
        rc = osp_result_copy(res, reinterpret_cast<uint64_t *>(out.pos.data()), out.data.data());
        osp_result_free(res);
        check(rc, ctx_, "coo2csr (device): copy");
        return out;
    }

private:
    osp_ctx *ctx_;
    osp_coo *h_;
};

class Engine {
public:
    explicit Engine(int device = 0) { check(osp_create(device, &ctx_), nullptr, "osp_create"); }
    ~Engine() { osp_destroy(ctx_); }
    Engine(const Engine &) = delete;
    Engine &operator=(const Engine &) = delete;
    osp_ctx *ctx() const { return ctx_; }

    // C = A * B; A as CSC (the reference's lmatCSC) unless a_is_csr.  rows_c = 0: numRows = max row id + 1.
    CSRMatrix spgemm(const CSRMatrix &a, const CSRMatrix &b, bool a_is_csr = false, size_t rows_c = 0, size_t cols_b = 0,
                     osp_stats *stats = nullptr, std::vector<std::pair<uint32_t, uint32_t>> *mult_tasks = nullptr,
                     std::vector<std::pair<uint32_t, uint32_t>> *merge_tasks = nullptr) {
        osp_spgemm_args args{};
        args.a_slices = a.NRow();
        args.a_pos = reinterpret_cast<const uint64_t *>(a.pos.data());
        args.a_data = a.data.data();
        args.n_k = b.NRow();
        args.b_pos = reinterpret_cast<const uint64_t *>(b.pos.data());
        args.b_data = b.data.data();
        args.rows_c = rows_c;
        args.cols_b = cols_b;
        args.flags = a_is_csr ? OSP_A_IS_CSR : 0u;
        osp_result *res = nullptr;
        check(osp_spgemm(ctx_, &args, &res), ctx_, "osp_spgemm");
        CSRMatrix c;
        try {
            uint64_t rows = 0, nnz = 0;
            osp_result_dims(res, &rows, &nnz);
            c.pos.resize(rows + 1);
            c.data.resize(nnz);
            check(osp_result_copy(res, reinterpret_cast<uint64_t *>(c.pos.data()), c.data.data()), ctx_, "osp_result_copy");
            if (stats) osp_result_stats(res, stats);
            if (mult_tasks || merge_tasks) {
                uint64_t nm = 0, ng = 0;
                check(osp_task_sizes(ctx_, &args, res, &nm, nullptr, &ng, nullptr), ctx_, "osp_task_sizes");
                std::vector<uint32_t> m(2 * nm), g(2 * ng);
                check(osp_task_sizes(ctx_, &args, res, &nm, m.data(), &ng, g.data()), ctx_, "osp_task_sizes");
                if (mult_tasks) { mult_tasks->resize(nm); for (uint64_t i = 0; i < nm; i++) (*mult_tasks)[i] = {m[2 * i], m[2 * i + 1]}; }
                if (merge_tasks) { merge_tasks->resize(ng); for (uint64_t i = 0; i < ng; i++) (*merge_tasks)[i] = {g[2 * i], g[2 * i + 1]}; }
            }
        } catch (...) {
            osp_result_free(res);
            throw;
        }
        osp_result_free(res);
        return c;
    }

    // compactMulcsr (SimSpGEMM.cpp:247-263), merged: the compact operand is a triplet list, so it enters through the
    // device COO ingest (coo2csr + dupcheck on the GPU) and the product runs like any other.  rows_a = rows of A
    // (0: largest row id + 1).  The reference returns the unmerged partial products of every group; merging them in
    // group order (= ascending k inside every output row) gives exactly this result.
    CSRMatrix compactMulcsr(const CompactCOOMatrix &compact, const CSRMatrix &csr, size_t rows_a = 0) {
        const size_t n = compact.data.size();
        std::vector<uint32_t> r(n), c(n);
        std::vector<float> v(n);
        for (size_t i = 0; i < n; i++) {
            r[i] = compact.data[i].row; c[i] = compact.data[i].col; v[i] = compact.data[i].val;
            if (size_t(r[i]) + 1 > rows_a) rows_a = size_t(r[i]) + 1;
        }
        CSRMatrix a;
        a.pos.assign(rows_a + 1, 0);
        a.data.resize(n);
        int rc = osp_coo2csr_device(ctx_, n, r.data(), c.data(), v.data(), rows_a, csr.NRow(), 0, 0,
                                    reinterpret_cast<uint64_t *>(a.pos.data()), a.data.data());
        if (rc == OSP_ERR_DUPLICATE) throw(233);            // compactMulcsr's dupcheck, SimSpGEMM.cpp:260
        check(rc, ctx_, "compactMulcsr: ingest");
        return spgemm(a, csr, /*a_is_csr=*/true);
    }

    // readcoo(path, NRow, NCol, sym) with the text parsed on the device: the triplets stay in HBM
    DeviceCOO readcoo_device(const char *path, size_t &NRow, size_t &NCol, bool sym) {
        osp_coo *h = nullptr;
        check(osp_readcoo_device(ctx_, path, sym ? 1 : 0, &h), ctx_, "readcoo_device");
        uint64_t nr = 0, nc = 0;
        osp_coo_dims(h, &nr, &nc, nullptr);
        NRow = nr; NCol = nc;
        return DeviceCOO(ctx_, h);
    }

private:
    osp_ctx *ctx_ = nullptr;
};

inline Engine &default_engine() {
    static Engine e(0);
    return e;
}

// Sizes of one multiply task (MultiplyTask, SimOuterSPACE.cpp:34-37: lmatCol.size, rmatRow.size; every
// result row has rmatRow.size entries) and one merge task (MergeTask, :39-42: inputs.size(), output.size).
struct MultiplyTaskSize { index_t lmatCol, rmatRow; };
struct MergeTaskSize { index_t inputs, output; };

class TaskProvider {
public:
    TaskProvider(const CSRMatrix &lmatCSC, const CSRMatrix &rmatCSR, Engine *engine = nullptr) {
        if (lmatCSC.NRow() != rmatCSR.NRow())             // assert(lmat.NRow() == rmat.NRow()), SimOuterSPACE.cpp:47
            throw Error(OSP_ERR_INVALID, "TaskProvider: lmatCSC and rmatCSR must have the same number of slices");
        Engine &e = engine ? *engine : default_engine();
        std::vector<std::pair<uint32_t, uint32_t>> mt, gt;
        mergedResult = e.spgemm(lmatCSC, rmatCSR, false, 0, 0, &stats, &mt, &gt);
        multTasks.reserve(mt.size());
        for (auto &p : mt) multTasks.push_back(MultiplyTaskSize{p.first, p.second});
        mergeTasks.reserve(gt.size());
        for (auto &p : gt) mergeTasks.push_back(MergeTaskSize{p.first, p.second});
    }
    const std::vector<MultiplyTaskSize> &getMultiplyTasks() { return multTasks; }
    const std::vector<MergeTaskSize> &getMergeTasks() { return mergeTasks; }

    CSRMatrix mergedResult;      // private and wrong-valued in the reference (SURVEY.md 8a rows a11/a12)
    osp_stats stats{};

private:
    std::vector<MultiplyTaskSize> multTasks;
    std::vector<MergeTaskSize> mergeTasks;
};

}  // namespace osp_b200

#endif  // OSP_B200_HPP
