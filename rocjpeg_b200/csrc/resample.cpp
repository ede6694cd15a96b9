// resample.cpp — see resample.h. Restates precompute_coeffs and normalize_coeffs_8bpc of Pillow's
// src/libImaging/Resample.c, filter functions included, operation for operation.
#include "resample.h"

#include <cmath>
#include <vector>

namespace rjb {

namespace {

double BoxFilter(double x) { return (x > -0.5 && x <= 0.5) ? 1.0 : 0.0; }

double BilinearFilter(double x) {
    if (x < 0.0) x = -x;
    return x < 1.0 ? 1.0 - x : 0.0;
}

double HammingFilter(double x) {
    if (x < 0.0) x = -x;
    if (x == 0.0) return 1.0;
    if (x >= 1.0) return 0.0;
    x = x * M_PI;
    // Pillow writes the window's constants as float literals (0.54f, 0.46f), promoted to double: with 0.54 and 0.46 some
    // 22-bit weights round one unit apart from Pillow's
    return std::sin(x) / x * (double(0.54f) + double(0.46f) * std::cos(x));
}

double BicubicFilter(double x) {
    const double a = -0.5;   // Pillow's bicubic parameter
    if (x < 0.0) x = -x;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}

double SincFilter(double x) {
    if (x == 0.0) return 1.0;
    x = x * M_PI;
    return std::sin(x) / x;
}

double LanczosFilter(double x) { return (-3.0 <= x && x < 3.0) ? SincFilter(x) * SincFilter(x / 3) : 0.0; }

struct Filter {
    double (*fn)(double);
    double support;
};

Filter FilterOf(int filter) {
    switch (filter) {
        case kFilterBox: return {BoxFilter, 0.5};
        case kFilterBilinear: return {BilinearFilter, 1.0};
        case kFilterHamming: return {HammingFilter, 1.0};
        case kFilterBicubic: return {BicubicFilter, 2.0};
        default: return {LanczosFilter, 3.0};
    }
}

double Support(uint32_t in_size, uint32_t out_size, const Filter& f, double* scale, double* filterscale) {
    *scale = double(in_size) / double(out_size);
    *filterscale = *scale < 1.0 ? 1.0 : *scale;
    return f.support * *filterscale;
}

}  // namespace

int ResizeTaps(uint32_t in_size, uint32_t out_size, int filter) {
    double scale, filterscale;
    const double support = Support(in_size, out_size, FilterOf(filter), &scale, &filterscale);
    return int(std::ceil(support)) * 2 + 1;
}

void ResizeCoefficients(uint32_t in_size, uint32_t out_size, int filter, int32_t* bounds, int32_t* taps) {
    const Filter f = FilterOf(filter);
    double scale, filterscale;
    const double support = Support(in_size, out_size, f, &scale, &filterscale);
    const int ksize = int(std::ceil(support)) * 2 + 1;
    const double ss = 1.0 / filterscale;
    std::vector<double> k(size_t(ksize), 0.0);   // weights of one output sample before rounding
    for (uint32_t xx = 0; xx < out_size; xx++) {
        const double center = (xx + 0.5) * scale;
        int xmin = int(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = int(center + support + 0.5);
        if (xmax > int(in_size)) xmax = int(in_size);
        xmax -= xmin;
        double ww = 0.0;
        for (int x = 0; x < xmax; x++) {
            const double w = f.fn((x + xmin - center + 0.5) * ss);
            k[x] = w;
            ww += w;
        }
        for (int x = 0; x < xmax; x++)
            if (ww != 0.0) k[x] /= ww;
        int32_t* kk = taps + size_t(xx) * size_t(ksize);
        for (int x = 0; x < ksize; x++) {
            const double v = x < xmax ? k[x] : 0.0;
            kk[x] = v < 0 ? int32_t(-0.5 + v * (1 << kResamplePrecision)) : int32_t(0.5 + v * (1 << kResamplePrecision));
        }
        bounds[2 * xx] = xmin;
        bounds[2 * xx + 1] = xmax;
    }
}

}  // namespace rjb
