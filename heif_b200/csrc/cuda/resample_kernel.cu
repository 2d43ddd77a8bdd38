// Stage 7 (optional, inside HEIC_STAGE_COLOR): resampling of the colour stage's RGB8 to any size, byte-equal to Pillow's
// Image.resize (include/heic_b200.h, heic_b200_decode_grids_resized).  Two separable passes, each pure int32 arithmetic
// on host-built fixed-point tables: per channel s = 2^21 + sum in[xmin + x] * k[x], out = clamp(s >> 22, 0, 255).
//
// The passes are not fused: Pillow clips the horizontal result to uint8 before the vertical pass reads it, and a fused
// kernel would have to recompute every intermediate row for each of the ~2 * support * fs output rows that read it.
#include <cuda_runtime.h>

#include <algorithm>

#include "kernels.h"

namespace heic {
namespace dev {

namespace {

constexpr int kHThreads = 256;                      // kResampleBand output columns x kHRows rows
constexpr int kHRows = kHThreads / kResampleBand;   // rows a CTA computes at once (one per warp)
constexpr int kHRowsPerCta = 32;                    // rows a CTA walks through with one load of its band's coefficients
constexpr int kVThreads = 128;                      // a thread writes 16 bytes of an output row
constexpr uint32_t kHMaxSmem = 200 * 1024;          // above this a band takes resample_h_wide_kernel (sm_100: 227 KB)

__device__ __forceinline__ uint32_t out8(int s) { return (uint32_t)min(255, max(0, s >> 22)); }

// A CTA takes one band of kResampleBand output columns of one image over kHRowsPerCta rows.  The band's coefficients
// (tap-major, so that the 32 lanes read 32 consecutive words) stay in shared memory for all its rows; the input span of
// kHRows rows at a time is copied in with 16-byte loads.  A thread computes one output pixel: three int32 accumulators,
// one IMAD per tap and channel.  Every output of the band runs the band's largest tap count: the taps past an output's
// own n have coefficient 0 and read whatever lies in the row buffer there.
__global__ void __launch_bounds__(kHThreads) resample_h_kernel(ResampleJob J, ResampleAxis A, uint32_t row_chunks) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint32_t b = blockIdx.x;
  const uint32_t chunk = b % row_chunks;
  b /= row_chunks;
  const uint32_t band = b % A.n_bands, image = b / A.n_bands;
  const int4 bd = A.band[band];
  const uint32_t taps = (uint32_t)bd.z;
  int32_t* sk = reinterpret_cast<int32_t*>(smem);
  uint8_t* srow = smem + (size_t)A.max_taps * kResampleBand * 4;
  const uint4* gk = reinterpret_cast<const uint4*>(A.coeffs + bd.w);
  for (uint32_t i = threadIdx.x; i < taps * (kResampleBand / 4); i += kHThreads) reinterpret_cast<uint4*>(sk)[i] = gk[i];
  const uint32_t lane = threadIdx.x % kResampleBand, warp = threadIdx.x / kResampleBand;
  const uint32_t j = band * kResampleBand + lane;
  const bool valid = j < A.n_out;
  const int4 o = A.out[valid ? j : band * kResampleBand];
  // the span's bytes [a0, a1) of a source row, 16-byte aligned (the source pitch is a multiple of 16 and covers a1)
  const uint32_t a0 = (3u * (uint32_t)bd.x) & ~15u, a1 = (3u * (uint32_t)(bd.x + bd.y) + 15u) & ~15u;
  const uint32_t n16 = (a1 - a0) >> 4;
  const uint32_t first = (3u * (uint32_t)o.x) - a0;  // this output's tap 0 inside a row buffer
  const uint8_t* img = J.src + (size_t)image * J.src_image_stride + (size_t)J.row0 * J.src_pitch + a0;
  uint8_t* dimg = J.dst + (size_t)image * J.dst_image_stride + (size_t)j * 3;
  const uint32_t r_end = min(J.rows, (chunk + 1) * kHRowsPerCta);
  for (uint32_t r0 = chunk * kHRowsPerCta; r0 < r_end; r0 += kHRows) {
    __syncthreads();  // the coefficients are in; the previous rows are consumed
    for (uint32_t q = threadIdx.x; q < kHRows * n16; q += kHThreads) {
      const uint32_t r = q / n16, c = q - r * n16;
      if (r0 + r < r_end)
        reinterpret_cast<uint4*>(srow + r * A.max_row_bytes)[c] =
            reinterpret_cast<const uint4*>(img + (size_t)(r0 + r) * J.src_pitch)[c];
    }
    __syncthreads();
    const uint32_t row = r0 + warp;
    if (row < r_end && valid) {
      const uint8_t* p = srow + warp * A.max_row_bytes + first;
      int s0 = 1 << 21, s1 = 1 << 21, s2 = 1 << 21;
      for (uint32_t x = 0; x < taps; x++) {
        const int k = sk[x * kResampleBand + lane];
        s0 += (int)p[3 * x] * k;
        s1 += (int)p[3 * x + 1] * k;
        s2 += (int)p[3 * x + 2] * k;
      }
      uint8_t* d = dimg + (size_t)row * J.dst_pitch;
      d[0] = (uint8_t)out8(s0);
      d[1] = (uint8_t)out8(s1);
      d[2] = (uint8_t)out8(s2);
    }
  }
}

// The same from global memory, for bands whose coefficients and span do not fit shared memory (extreme ratios: output j
// of 4032 -> 1 under Lanczos reads the whole row).  Correct, not fast: each thread runs its own n taps.
__global__ void __launch_bounds__(kHThreads) resample_h_wide_kernel(ResampleJob J, ResampleAxis A, uint32_t row_groups) {
  uint32_t b = blockIdx.x;
  const uint32_t rg = b % row_groups;
  b /= row_groups;
  const uint32_t band = b % A.n_bands, image = b / A.n_bands;
  const uint32_t lane = threadIdx.x % kResampleBand, warp = threadIdx.x / kResampleBand;
  const uint32_t j = band * kResampleBand + lane, row = rg * kHRows + warp;
  if (j >= A.n_out || row >= J.rows) return;
  const int4 o = A.out[j];
  const uint8_t* p = J.src + (size_t)image * J.src_image_stride + (size_t)(J.row0 + row) * J.src_pitch + (size_t)o.x * 3;
  const int32_t* k = A.coeffs + o.z;
  int s0 = 1 << 21, s1 = 1 << 21, s2 = 1 << 21;
  for (int x = 0; x < o.y; x++) {
    const int kx = __ldg(k + (size_t)x * kResampleBand);
    s0 += (int)p[3 * x] * kx;
    s1 += (int)p[3 * x + 1] * kx;
    s2 += (int)p[3 * x + 2] * kx;
  }
  uint8_t* d = J.dst + (size_t)image * J.dst_image_stride + (size_t)row * J.dst_pitch + (size_t)j * 3;
  d[0] = (uint8_t)out8(s0);
  d[1] = (uint8_t)out8(s1);
  d[2] = (uint8_t)out8(s2);
}

__device__ __forceinline__ void mac4(int (&s)[16], int base, uint32_t w, int k) {
  s[base + 0] += (int)(w & 0xffu) * k;
  s[base + 1] += (int)((w >> 8) & 0xffu) * k;
  s[base + 2] += (int)((w >> 16) & 0xffu) * k;
  s[base + 3] += (int)(w >> 24) * k;
}

__device__ __forceinline__ uint32_t pack_out(const int (&s)[16], int base) {
  return out8(s[base]) | (out8(s[base + 1]) << 8) | (out8(s[base + 2]) << 16) | (out8(s[base + 3]) << 24);
}

// Vertical pass: channels are independent along y, so a thread takes 16 consecutive bytes of an output row (5 1/3
// pixels): one 16-byte load per tap from rows that the warp reads coalesced across x, 16 IMADs, one 16-byte store.  The
// rows are 16-byte aligned and their pitch a multiple of 16, so a row's last 16 bytes may run into its padding, never
// past it.  Every thread of a CTA works on the same output row: the coefficient loads are uniform.
__global__ void __launch_bounds__(kVThreads) resample_v_kernel(ResampleJob J, ResampleAxis A) {
  const uint32_t c = blockIdx.x * kVThreads + threadIdx.x, yy = blockIdx.y, image = blockIdx.z;
  if (c * 16 >= J.out_w * 3) return;
  const int4 o = A.out[yy];
  const uint8_t* p = J.src + (size_t)image * J.src_image_stride + (size_t)(o.x - (int)J.row0) * J.src_pitch + (size_t)c * 16;
  const int32_t* k = A.coeffs + o.z;
  int s[16];
#pragma unroll
  for (int i = 0; i < 16; i++) s[i] = 1 << 21;
  for (int y = 0; y < o.y; y++) {
    const int ky = __ldg(k + (size_t)y * kResampleBand);
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p + (size_t)y * J.src_pitch));
    mac4(s, 0, v.x, ky);
    mac4(s, 4, v.y, ky);
    mac4(s, 8, v.z, ky);
    mac4(s, 12, v.w, ky);
  }
  *reinterpret_cast<uint4*>(J.dst + (size_t)image * J.dst_image_stride + (size_t)yy * J.dst_pitch + (size_t)c * 16) =
      make_uint4(pack_out(s, 0), pack_out(s, 4), pack_out(s, 8), pack_out(s, 12));
}

}  // namespace

cudaError_t launch_resample_h(const ResampleJob& job, const ResampleAxis& ax, cudaStream_t stream) {
  if (!job.n_images || !job.rows || !ax.n_out) return cudaSuccess;
  const size_t smem = (size_t)ax.max_taps * kResampleBand * 4 + (size_t)kHRows * ax.max_row_bytes;
  if (smem <= kHMaxSmem) {
    // per device, so on every launch (a process may drive several GPUs)
    const cudaError_t attr = cudaFuncSetAttribute(resample_h_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHMaxSmem);
    if (attr != cudaSuccess) return attr;
    const uint32_t row_chunks = (job.rows + kHRowsPerCta - 1) / kHRowsPerCta;
    const unsigned grid = job.n_images * ax.n_bands * row_chunks;
    resample_h_kernel<<<grid, kHThreads, smem, stream>>>(job, ax, row_chunks);
  } else {
    const uint32_t row_groups = (job.rows + kHRows - 1) / kHRows;
    const unsigned grid = job.n_images * ax.n_bands * row_groups;
    resample_h_wide_kernel<<<grid, kHThreads, 0, stream>>>(job, ax, row_groups);
  }
  return cudaGetLastError();
}

cudaError_t launch_resample_v(const ResampleJob& job, const ResampleAxis& ax, cudaStream_t stream) {
  if (!job.n_images || !job.rows || !job.out_w) return cudaSuccess;
  const uint32_t chunks = (job.out_w * 3 + 15) / 16;
  for (uint32_t i0 = 0; i0 < job.n_images; i0 += 65535) {  // gridDim.z limit
    ResampleJob j = job;
    j.src += (size_t)i0 * job.src_image_stride;
    j.dst += (size_t)i0 * job.dst_image_stride;
    j.n_images = std::min(job.n_images - i0, 65535u);
    const dim3 grid((chunks + kVThreads - 1) / kVThreads, j.rows, j.n_images);
    resample_v_kernel<<<grid, kVThreads, 0, stream>>>(j, ax);
  }
  return cudaGetLastError();
}

}  // namespace dev
}  // namespace heic
