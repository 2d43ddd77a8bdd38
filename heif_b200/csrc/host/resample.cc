// Coefficient tables of the resampling stage: a restatement of Pillow's precompute_coeffs and normalize_coeffs_8bpc
// (libImaging/Resample.c) in IEEE double, evaluated on the host.  Only these tables involve floating point; the passes
// that use them are integer arithmetic.  The tables are built here rather than on the device because nvcc contracts
// a * b + c into a fused multiply-add by default, which changes the doubles; sin and cos come from the host C library,
// as Pillow's do.  The optimize attribute keeps the host compiler from contracting either (it would on targets with FMA).
#include "resample.h"

#include <cmath>
#include <cstring>

#include "capi_common.h"

namespace heic {
namespace {

#define HEIC_NO_CONTRACT __attribute__((optimize("fp-contract=off")))

HEIC_NO_CONTRACT double box_filter(double x) { return (x > -0.5 && x <= 0.5) ? 1.0 : 0.0; }

HEIC_NO_CONTRACT double bilinear_filter(double x) {
  if (x < 0.0) x = -x;
  return x < 1.0 ? 1.0 - x : 0.0;
}

HEIC_NO_CONTRACT double hamming_filter(double x) {
  if (x < 0.0) x = -x;
  if (x == 0.0) return 1.0;
  if (x >= 1.0) return 0.0;
  x = x * M_PI;
  // Pillow writes the window's constants as float literals: 0.54f and 0.46f, widened to double
  return std::sin(x) / x * (0.54f + 0.46f * std::cos(x));
}

HEIC_NO_CONTRACT double bicubic_filter(double x) {
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}

HEIC_NO_CONTRACT double sinc_filter(double x) {
  if (x == 0.0) return 1.0;
  x = x * M_PI;
  return std::sin(x) / x;
}

HEIC_NO_CONTRACT double lanczos_filter(double x) {
  if (-3.0 <= x && x < 3.0) return sinc_filter(x) * sinc_filter(x / 3);
  return 0.0;
}

struct Filter {
  double (*fn)(double);
  double support;
};

// indexed by HEIC_RESAMPLE_* (Pillow's Image.Resampling numbers; 0 is NEAREST, which is not a filter of this path)
const Filter kFilters[6] = {{nullptr, 0.0},         {lanczos_filter, 3.0}, {bilinear_filter, 1.0},
                            {bicubic_filter, 2.0},  {box_filter, 0.5},     {hamming_filter, 1.0}};

}  // namespace

HEIC_NO_CONTRACT void resample_coeffs(uint32_t n_in, uint32_t n_out, uint32_t filter, ResampleTable& t) {
  if (!n_in || n_in > (1u << 24) || !n_out || n_out > kResampleMaxSide || filter < 1 || filter > 5)
    bail(HEIC_E_INVALID_ARG, "resample: input side 0 or above 2^24, output side outside 1..32768, or filter outside 1..5");
  const Filter& f = kFilters[filter];
  double scale = (double)n_in / n_out, filterscale = scale;
  if (filterscale < 1.0) filterscale = 1.0;
  const double support = f.support * filterscale;
  const size_t ksize = (size_t)std::ceil(support) * 2 + 1;
  t.xmin.assign(n_out, 0);
  t.n.assign(n_out, 0);
  t.off.assign(n_out + 1, 0);
  t.coeffs.clear();
  std::vector<double> k(ksize);
  for (uint32_t xx = 0; xx < n_out; xx++) {
    const double center = (xx + 0.5) * scale;
    const double ss = 1.0 / filterscale;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > (int)n_in) xmax = (int)n_in;
    xmax -= xmin;
    double ww = 0.0;
    for (int x = 0; x < xmax; x++) {
      const double w = f.fn((x + xmin - center + 0.5) * ss);
      k[x] = w;
      ww += w;
    }
    for (int x = 0; x < xmax; x++)
      if (ww != 0.0) k[x] /= ww;
    t.xmin[xx] = xmin;
    t.n[xx] = xmax;
    t.off[xx] = (uint32_t)t.coeffs.size();
    for (int x = 0; x < xmax; x++)
      t.coeffs.push_back(k[x] < 0 ? (int32_t)(-0.5 + k[x] * (1 << kResamplePrecisionBits))
                                  : (int32_t)(0.5 + k[x] * (1 << kResamplePrecisionBits)));
  }
  t.off[n_out] = (uint32_t)t.coeffs.size();
}

}  // namespace heic

using namespace heic;

extern "C" int64_t heic_b200_resample_coeffs(uint32_t n_in, uint32_t n_out, uint32_t filter, int32_t* bounds, int32_t* coeffs,
                                             size_t coeffs_cap) {
  return guard([&]() -> int64_t {
    ResampleTable t;
    resample_coeffs(n_in, n_out, filter, t);
    if (coeffs && coeffs_cap < t.coeffs.size()) bail(HEIC_E_INVALID_ARG, "resample: coefficient buffer too small");
    if (bounds)
      for (uint32_t j = 0; j < n_out; j++) bounds[2 * j] = t.xmin[j], bounds[2 * j + 1] = t.n[j];
    if (coeffs) std::memcpy(coeffs, t.coeffs.data(), t.coeffs.size() * sizeof(int32_t));
    return (int64_t)t.coeffs.size();
  });
}
