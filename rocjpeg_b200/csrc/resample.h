// resample.h — Pillow's resampling filters restated on the host: the tables the resize passes (k4_resize.cu) apply.
//
// Pillow (src/libImaging/Resample.c) resizes with a separable filter whose weights it computes in double precision
// (precompute_coeffs) and rounds to fixed point with 22 fractional bits (normalize_coeffs_8bpc); both passes are then
// int32 multiply-adds that start at 1 << 21 and clip `acc >> 22` to 0..255. The same doubles, the same libm sin / cos
// and the same rounding here make the GPU passes byte-identical to Image.resize.
#pragma once
#include <stdint.h>

namespace rjb {

// Pillow's Image.Resampling values (ROCJPEG_B200_FILTER_* of include/rocjpeg_b200_ext.h); NEAREST (0) is not a filter here
enum ResampleFilter : int32_t { kFilterLanczos = 1, kFilterBilinear = 2, kFilterBicubic = 3, kFilterBox = 4, kFilterHamming = 5 };
constexpr int kResamplePrecision = 22;   // fractional bits of the fixed-point weights
constexpr uint32_t kMaxResizeSize = 65535;

inline bool ValidFilter(int f) { return f >= kFilterLanczos && f <= kFilterHamming; }

// Taps per output sample Pillow reserves for an axis resized from in_size to out_size: 2 * ceil(support) + 1.
int ResizeTaps(uint32_t in_size, uint32_t out_size, int filter);

// Pillow's coefficients of one axis: bounds[2 i] = first input sample of output sample i, bounds[2 i + 1] = how many it
// reads (at most the taps per sample); taps[i * ksize + t] = fixed-point weight of input sample bounds[2 i] + t (rows
// padded with zeros to ksize = ResizeTaps(...)). Sizes >= 1, a valid filter.
void ResizeCoefficients(uint32_t in_size, uint32_t out_size, int filter, int32_t* bounds, int32_t* taps);

}  // namespace rjb
