// osp_spgemm_cli -- the reference's command line (simulator/SimSpGEMM.cpp:819-894) on the GPU engine:
//
//     osp_spgemm_cli A.mtx B.mtx [--no-transpose] [--dump out.mtx] [--device-ingest]
//
// reads two Matrix-Market files, transposes matrix 2 (the reference's "Workaround: Transpose Matrix 2",
// :852-856, so the product is F1 * F2^T), builds CSC(F1) and CSR(F2^T) with coo2csr, prints the same
// dimension / "mul flops ref" lines, then runs TaskProvider (multiply + merge) on the B200 instead of the
// CPU and prints the result size, an FNV-1a checksum of C (pos + data bytes) and GFLOP/s (2 flops per
// product).  The cycle-level simulator (simulateOuterSPACE) is not part of this tool: it stays in the
// reference and can be fed from getMultiplyTasks()/getMergeTasks().
// --device-ingest parses both files on the GPU (osp_readcoo_device) and builds CSC(F1) and CSR(F2^T) there
// (osp_coo2csr_result; the transpose of matrix 2 is coo2csr<true> of its triplets), then copies them back for the same
// TaskProvider: every line is the same except the timing lines, plus one line with the ingest time.
#include <chrono>
#include <cstdio>
#include <cstring>
#include <fstream>

#include "../include/osp_b200.hpp"

using namespace osp_b200;

static uint64_t fnv1a(const void *p, size_t n, uint64_t h) {
    const unsigned char *b = static_cast<const unsigned char *>(p);
    for (size_t i = 0; i < n; i++) { h ^= b[i]; h *= 1099511628211ull; }
    return h;
}

int main(int argc, char **argv) {
    if (argc < 3) {
        std::fprintf(stderr, "usage: %s A.mtx B.mtx [--no-transpose] [--dump out.mtx] [--device-ingest]\n", argv[0]);
        return 2;
    }
    bool transpose2 = true, device_ingest = false;
    const char *dump = nullptr;
    for (int i = 3; i < argc; i++) {
        if (!std::strcmp(argv[i], "--no-transpose")) transpose2 = false;
        else if (!std::strcmp(argv[i], "--dump") && i + 1 < argc) dump = argv[++i];
        else if (!std::strcmp(argv[i], "--device-ingest")) device_ingest = true;
    }
    try {
        size_t NRow[2], NCol[2], nnz[2];
        CSRMatrix csc, csr;
        Engine eng(0);
        if (device_ingest) {
            auto t0 = std::chrono::high_resolution_clock::now();
            DeviceCOO d0 = eng.readcoo_device(argv[1], NRow[0], NCol[0], false);
            DeviceCOO d1 = eng.readcoo_device(argv[2], NRow[1], NCol[1], false);
            nnz[0] = d0.size(); nnz[1] = d1.size();
            if (transpose2) std::swap(NRow[1], NCol[1]);
            for (int i = 0; i < 2; i++)
                std::printf("NCol = %zu, NRow = %zu, NNZ = %zu\n", NRow[i], NCol[i], nnz[i]);
            csc = d0.coo2csr<true>(NCol[0]);
            csr = transpose2 ? d1.coo2csr<true>(NRow[1]) : d1.coo2csr<false>(NRow[1]);
            double sec = std::chrono::duration<double>(std::chrono::high_resolution_clock::now() - t0).count();
            std::printf("ingest on the device: %.3f ms (both files to CSC(F1) and CSR(F2^T), copied to the host)\n", sec * 1e3);
        } else {
            COOMatrix coo[2];
            for (int i = 0; i < 2; i++) {
                std::ifstream fin(argv[1 + i]);
                if (!fin) { std::fprintf(stderr, "cannot open %s\n", argv[1 + i]); return 1; }
                coo[i] = readcoo(fin, NRow[i], NCol[i], false);
                nnz[i] = coo[i].size();
            }
            if (transpose2) {
                std::swap(NRow[1], NCol[1]);
                for (auto &e : coo[1]) std::swap(e.row, e.col);
            }
            for (int i = 0; i < 2; i++)   // label order as printed by the reference (:866)
                std::printf("NCol = %zu, NRow = %zu, NNZ = %zu\n", NRow[i], NCol[i], nnz[i]);
            csc = coo2csr<true>(coo[0], NCol[0]);
            csr = coo2csr(coo[1], NRow[1]);
        }
        if (csr.pos.size() != csc.pos.size()) { std::fprintf(stderr, "inner dimensions differ\n"); return 1; }
        size_t flops = mulflops(csc, csr);
        std::printf("mul flops ref = %zu\n", flops);
        TaskProvider warm(csc, csr, &eng);                      // first call pays allocation / module load
        auto t0 = std::chrono::high_resolution_clock::now();
        TaskProvider provider(csc, csr, &eng);
        double sec = std::chrono::duration<double>(std::chrono::high_resolution_clock::now() - t0).count();
        const CSRMatrix &c = provider.mergedResult;
        uint64_t h = 1469598103934665603ull;
        h = fnv1a(c.pos.data(), c.pos.size() * sizeof(size_t), h);
        h = fnv1a(c.data.data(), c.data.size() * sizeof(CSRElement), h);
        std::printf("C rows = %zu, nnz = %zu, checksum = %016llx\n", c.NRow(), c.data.size(), (unsigned long long)h);
        std::printf("multiply tasks = %zu, merge tasks = %zu\n", provider.getMultiplyTasks().size(), provider.getMergeTasks().size());
        std::printf("B200 TaskProvider: %.3f ms host-to-host (device %.3f ms), %.2f GFlops (2 flops per product)\n", sec * 1e3,
                    provider.stats.ms_total, 2.0 * flops / sec * 1e-9);
        if (dump) {
            std::FILE *f = std::fopen(dump, "w");
            if (!f) { std::fprintf(stderr, "cannot write %s\n", dump); return 1; }
            size_t ncols = transpose2 ? NCol[1] : NCol[1];
            std::fprintf(f, "%%%%MatrixMarket matrix coordinate real general\n%zu %zu %zu\n", c.NRow(), ncols, c.data.size());
            for (size_t i = 0; i < c.NRow(); i++)
                for (size_t e = c.pos[i]; e < c.pos[i + 1]; e++)
                    std::fprintf(f, "%zu %u %.9g\n", i + 1, c.data[e].idx + 1, c.data[e].val);
            std::fclose(f);
        }
    } catch (int code) {
        std::fprintf(stderr, "error: duplicate entry (%d)\n", code);
        return 1;
    } catch (const std::exception &e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
