// osp_mtx_grammar.h -- the plain-line grammar of the .mtx loaders, compiled for the host (osp_host.cpp, g++) and for
// the device (osp_mtx.cuh, nvcc), so that the host and the device parser read every line the same way.
//
// A line of the plain shape  <digits> <blanks> <digits> [<blanks> <decimal number>]  is parsed in place: the indices as
// at most 19 digits, the value by Clinger's exact fast path (at most 15 significant digits and |decimal exponent| <= 22:
// mantissa and power of ten are both exact doubles, so one multiply or divide rounds correctly -- the double strtod /
// "%lf" produce).  A multiply or divide of two doubles is correctly rounded on the device as well (the build has no
// -ftz and no --use_fast_math), so both compilers give the same bits.  Every other line is "slow": the host reads it
// through the C library (slow_line, osp_mtx_host.h).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define OSP_MTX_HD __host__ __device__ __forceinline__
#else
#define OSP_MTX_HD inline
#endif

namespace osp_mtx {

#define OSP_MTX_POW10 {1e0,  1e1,  1e2,  1e3,  1e4,  1e5,  1e6,  1e7,  1e8,  1e9,  1e10, 1e11, \
                       1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22}
const double kPow10[23] = OSP_MTX_POW10;
#if defined(__CUDACC__)
__constant__ double kPow10_dev[23] = OSP_MTX_POW10;      // the same table in the device's constant bank
#endif
#undef OSP_MTX_POW10

OSP_MTX_HD double pow10_exact(int e) {
#if defined(__CUDA_ARCH__)
    return kPow10_dev[e];
#else
    return kPow10[e];
#endif
}

OSP_MTX_HD bool is_blank(char ch) { return ch == ' ' || ch == '\t' || ch == '\r' || ch == '\v' || ch == '\f'; }

// <digits>: at most 19 of them (no overflow of uint64); false = not of the plain shape.
OSP_MTX_HD bool fast_u64(const char *&s, const char *end, uint64_t &out) {
    const char *q = s;
    uint64_t v = 0;
    while (q < end && *q >= '0' && *q <= '9' && q - s < 19) v = v * 10 + uint64_t(*q++ - '0');
    if (q == s || (q < end && *q >= '0' && *q <= '9')) return false;
    out = v;
    s = q;
    return true;
}

// [sign] digits [. digits] [e [sign] digits] with an exactly representable mantissa and power of ten.
OSP_MTX_HD bool fast_f64(const char *&s, const char *end, double &out) {
    const char *q = s;
    bool neg = false;
    if (q < end && (*q == '-' || *q == '+')) neg = *q++ == '-';
    uint64_t m = 0;
    int digits = 0, frac = 0;
    bool any = false;
    while (q < end && *q >= '0' && *q <= '9') {
        any = true;
        if (m || *q != '0') { if (++digits > 15) return false; m = m * 10 + uint64_t(*q - '0'); }
        q++;
    }
    if (q < end && *q == '.') {
        q++;
        while (q < end && *q >= '0' && *q <= '9') {
            any = true;
            if (m || *q != '0') { if (++digits > 15) return false; m = m * 10 + uint64_t(*q - '0'); }
            frac++;
            q++;
        }
    }
    if (!any) return false;
    int e10 = 0;
    if (q < end && (*q == 'e' || *q == 'E')) {
        const char *r = q + 1;
        bool eneg = false;
        if (r < end && (*r == '-' || *r == '+')) eneg = *r++ == '-';
        if (r < end && *r >= '0' && *r <= '9') {                 // otherwise the 'e' is not part of the number
            int ev = 0;
            while (r < end && *r >= '0' && *r <= '9') { if (ev > 10000) return false; ev = ev * 10 + (*r++ - '0'); }
            e10 = eneg ? -ev : ev;
            q = r;
        }
    }
    // what follows must end the number for strtod as well (hex floats "0x..", "1.5p3" and the like take the slow path)
    if (q < end && !is_blank(*q)) {
        const char ch = *q;
        if ((ch >= '0' && ch <= '9') || ch == '.' || ch == 'x' || ch == 'X' || ch == 'p' || ch == 'P') return false;
    }
    const int e = e10 - frac;
    double v = double(m);                                        // exact: m < 10^15 < 2^53
    if (m != 0) {
        if (e < -22 || e > 22) return false;
        v = e >= 0 ? v * pow10_exact(e) : v / pow10_exact(-e);
    }
    out = neg ? -v : v;
    s = q;
    return true;
}

// What one line [q, le) (without its '\n') holds.  q is moved past the leading blanks: a slow line is read from there.
enum LineKind { LINE_SKIP = 0, LINE_ENTRY = 1, LINE_SLOW = 2 };
OSP_MTX_HD int plain_line(const char *&q, const char *le, uint64_t &r, uint64_t &col, double &v) {
    while (q < le && (*q == ' ' || *q == '\t' || *q == '\r')) q++;       // blank and '%' lines (SimSpGEMM.cpp:66-77; '\r' for CRLF files)
    if (q == le || *q == '%') return LINE_SKIP;
    v = 1.0;
    const char *t = q;
    bool ok = fast_u64(t, le, r) && t < le && is_blank(*t);
    if (ok) {
        while (t < le && is_blank(*t)) t++;
        ok = fast_u64(t, le, col) && (t == le || is_blank(*t));
    }
    if (ok) {
        while (t < le && is_blank(*t)) t++;
        if (t < le) ok = fast_f64(t, le, v);                  // no third field: the value stays 1.0
    }
    return ok ? LINE_ENTRY : LINE_SLOW;
}

}  // namespace osp_mtx
