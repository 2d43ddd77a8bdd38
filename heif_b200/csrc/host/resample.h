// Coefficient tables of the resampling stage (include/heic_b200.h, heic_b200_decode_grids_resized): Pillow's
// precompute_coeffs + normalize_coeffs_8bpc (Resample.c), the only floating-point part of Image.resize.
#pragma once
#include <cstdint>
#include <vector>

namespace heic {

constexpr uint32_t kResampleMaxSide = 32768;  // largest resized side the library accepts
constexpr int kResamplePrecisionBits = 22;    // Pillow's PRECISION_BITS for 8-bit images (32 - 8 - 2)

// One axis n_in -> n_out under a filter (HEIC_RESAMPLE_*): output j reads input samples [xmin[j], xmin[j] + n[j]) with the
// fixed-point weights coeffs[off[j] .. off[j] + n[j]).
struct ResampleTable {
  std::vector<int32_t> xmin, n;
  std::vector<uint32_t> off;  // n_out + 1 entries: the taps are packed back to back
  std::vector<int32_t> coeffs;
};

// Throws HEIC_E_INVALID_ARG for n_in = 0, n_out outside 1..kResampleMaxSide or an unknown filter.
void resample_coeffs(uint32_t n_in, uint32_t n_out, uint32_t filter, ResampleTable& t);

}  // namespace heic
