// osp_mtx_host.h -- what the host loaders (osp_host.cpp) share with the device ingest of osp_engine.cu: the osp_coo
// handle, the header line and the C-library reading of a slow line.  Internal: not part of the C ABI.
#pragma once
#include "../../include/osp_b200.h"

#include <string>
#include <vector>

// Triplets of one .mtx file, on the host (osp_readcoo) or in HBM of ctx (osp_readcoo_device: ctx != NULL).
struct osp_coo {
    uint64_t nrow = 0, ncol = 0, nnz_header = 0;
    std::vector<uint32_t> rows, cols;
    std::vector<float> vals;
    osp_ctx *ctx = nullptr;
    uint32_t *d_rows = nullptr, *d_cols = nullptr;
    float *d_vals = nullptr;
    uint64_t d_nnz = 0;
    uint32_t max_row = 0, max_col = 0;            // largest stored row and col id (device triplets, nnz > 0)
};

namespace osp_mtx {

struct Piece {
    std::vector<uint32_t> rows, cols;
    std::vector<float> vals;
    int err = OSP_OK;
};

// One line of text (without its '\n'): false for a blank or '%' line; otherwise the header "NRow NCol NNZ" is read
// into hdr the way sscanf("%zu %zu %zu") reads it (SimSpGEMM.cpp:66-88) and the result is true.
bool header_line(const std::string &line, uint64_t hdr[3]);

// The reference's behaviour on any line, through the C library: appends its one or two entries to out.
int slow_line(const std::string &line, int symmetric, Piece &out);

}  // namespace osp_mtx

// Device-resident osp_coo (osp_engine.cu).
int osp_coo_device_copy(const osp_coo *c, uint32_t *rows, uint32_t *cols, float *vals);
void osp_coo_device_free(osp_coo *c);
