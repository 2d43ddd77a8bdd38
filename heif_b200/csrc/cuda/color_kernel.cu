// Stage 6: YCbCr 4:2:0 -> RGB8 fused with HEIF grid stitching, conformance windows, the canvas crop and the output geometry
// (clap crop, irot turns, imir mirrors) — one bandwidth-bound pass: 1.5 B read + 3 B written per output pixel.  Unturned,
// uncropped rows leave through shared memory as bulk copies (TMA, cp.async.bulk: UBLKCP in SASS); every other geometry is
// laid down in output orientation in shared memory.
//
// The reference's src/color is an ICC-header stub, not a converter (SURVEY 0.3), so the conversion is the
// frozen integer definition of SURVEY row C1 (libheif-style nearest-neighbour chroma, 8.8 fixed point):
//   full range BT.601:  R = clip8(Y + ((359 d + 128) >> 8)),  G = clip8(Y + ((-88 c - 183 d + 128) >> 8)),
//                       B = clip8(Y + ((454 c + 128) >> 8)),  c = Cb - 128, d = Cr - 128
// with the BT.709 / limited-range variants listed in oracle/hevc_oracle.c (color_coeffs).
#include <cuda_runtime.h>

#include "kernels.h"

namespace heic {
namespace dev {

namespace {

struct Coeffs {
  int y_mul, y_sub, rv, gu, gv, bu;
};

__device__ __forceinline__ uint32_t clip8(int v) { return (uint32_t)min(255, max(0, v)); }

__device__ __forceinline__ uint32_t pack4(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  return __byte_perm(__byte_perm(a, b, 0x0040), __byte_perm(c, d, 0x0040), 0x5410);
}

// One 16-byte store row of the staging buffer = 48 bytes of RGB per thread: a CTA's 128 threads lay down 6144 contiguous
// bytes per canvas row, which go to HBM as ONE bulk copy (TMA, cp.async.bulk shared -> global).
constexpr int kColorThreads = 128;
constexpr int kStageVec = kColorThreads * 3;  // uint4 per staged row

__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gdst), "r"(s), "r"(bytes) : "memory");
}

// A thread converts a 16 x 2 block of the canvas (two rows share one row of chroma): 32 + 16 bytes in, 96 bytes out.
// FULL: full-range input, where (256 Y + t) >> 8 == Y + (t >> 8): the chroma terms are computed once per 2x2 quad, and the
//   two pixels of a row that share them are clamped together by one VIADDMNMX.S16x2.RELU (max(min(Y + t, 255), 0) on both
//   16-bit halves), so a pixel costs half an instruction per channel plus the byte shuffles.
// FUSED: the planes are the deblocked reconstruction; CTBs with SAO on are read from the final arena (see convert_block).
// BULK: unrotated output whose rows are multiples of 16 bytes: the RGB of the CTA's strip is staged in shared memory and
//   stored by two bulk copies (one per row) instead of 3 x 16-byte stores per thread and row at a 48-byte stride.
// grid: flat over (image, pair of canvas rows, block of 16-pixel groups).
// RGB of the 16 x 2 block at canvas position (x, y) of `image` as 2 x 12 packed words (row r: w[r][0..11] = 48 bytes).
template <bool FULL, bool FUSED>
__device__ __forceinline__ void convert_block(const ColorJob& J, const Coeffs& K, uint32_t image, uint32_t x, uint32_t y, bool two_rows,
                                              uint32_t (&w)[2][12]) {
  const uint32_t tr = y / J.tile_h, ly = y - tr * J.tile_h;
  uint32_t yv[2][4], cbv[2], crv[2];
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const uint32_t xh = x + 8 * h;
    if (xh < J.out_w) {
      const uint32_t tc = xh / J.tile_w, lx = xh - tc * J.tile_w;
      const uint32_t ti = image * J.grid_cols * J.grid_rows + tr * J.grid_cols + tc;
      const uint8_t* t = J.planes + (size_t)ti * J.tile_stride;
      const uint8_t *ty = t, *tcb = t, *tcr = t;
      if (FUSED) {
        // the eight luma samples (both rows: ly is even) and the four chroma samples lie in one CTB; a component whose SAO
        // type is non-zero there has its final samples in the other arena (written by sao_sparse_kernel), every other one
        // is final as deblocked.  One 16-byte load of the CTB's parameter words decides (they are zero where SAO is off).
        const uint4 sp = *reinterpret_cast<const uint4*>(J.sao + (size_t)ti * J.sao_stride +
                                                         (size_t)((ly >> J.log2_ctb) * J.wctb + (lx >> J.log2_ctb)) * 4);
        const uint8_t* t2 = J.planes_sao + (size_t)ti * J.tile_stride;
        if (sp.x & 3u) ty = t2;
        if (sp.y & 3u) tcb = t2;
        if (sp.z & 3u) tcr = t2;
      }
      const uint2 a = *reinterpret_cast<const uint2*>(ty + (size_t)ly * J.pitch_y + lx);
      const uint2 b = two_rows ? *reinterpret_cast<const uint2*>(ty + (size_t)(ly + 1) * J.pitch_y + lx) : make_uint2(0u, 0u);
      cbv[h] = crv[h] = 0x80808080u;
      if (J.chroma) {
        const size_t co = (size_t)(ly >> 1) * J.pitch_c + (lx >> 1);
        cbv[h] = *reinterpret_cast<const uint32_t*>(tcb + J.cb_off + co);
        crv[h] = *reinterpret_cast<const uint32_t*>(tcr + J.cr_off + co);
      }
      yv[0][2 * h] = a.x, yv[0][2 * h + 1] = a.y, yv[1][2 * h] = b.x, yv[1][2 * h + 1] = b.y;
    } else {
      yv[0][2 * h] = yv[0][2 * h + 1] = yv[1][2 * h] = yv[1][2 * h + 1] = 0u;
      cbv[h] = crv[h] = 0x80808080u;
    }
  }
#pragma unroll
  for (int q = 0; q < 4; q++) {  // groups of four pixels -> three output words per row
    if (FULL) {
      uint32_t rg[2][2], bb[2][2];  // [row][pixel pair]: R | G << 8 and B of the two pixels in the 16-bit halves
#pragma unroll
      for (int jj = 0; jj < 2; jj++) {
        const int j = 2 * q + jj;  // chroma sample index 0..7
        const int c = (int)((cbv[j >> 2] >> (8 * (j & 3))) & 0xffu) - 128, d = (int)((crv[j >> 2] >> (8 * (j & 3))) & 0xffu) - 128;
        // the three chroma terms, each duplicated into both 16-bit halves
        const uint32_t r2 = __byte_perm((uint32_t)((K.rv * d + 128) >> 8), 0u, 0x1010);
        const uint32_t g2 = __byte_perm((uint32_t)((K.gu * c + K.gv * d + 128) >> 8), 0u, 0x1010);
        const uint32_t b2 = __byte_perm((uint32_t)((K.bu * c + 128) >> 8), 0u, 0x1010);
#pragma unroll
        for (int r = 0; r < 2; r++) {
          const uint32_t y2 = __byte_perm(yv[r][q], 0u, jj ? 0x4342 : 0x4140);  // Y of the pair's two pixels, zero-extended
          const uint32_t R = __viaddmin_s16x2_relu(y2, r2, 0x00ff00ffu), G = __viaddmin_s16x2_relu(y2, g2, 0x00ff00ffu);
          bb[r][jj] = __viaddmin_s16x2_relu(y2, b2, 0x00ff00ffu);
          rg[r][jj] = __byte_perm(R, G, 0x6240);  // R0 G0 R1 G1
        }
      }
#pragma unroll
      for (int r = 0; r < 2; r++) {
        w[r][3 * q + 0] = __byte_perm(rg[r][0], bb[r][0], 0x2410);                                     // R0 G0 B0 R1
        w[r][3 * q + 1] = __byte_perm(__byte_perm(rg[r][0], bb[r][0], 0x0063), rg[r][1], 0x5410);     // G1 B1 R2 G2
        w[r][3 * q + 2] = __byte_perm(bb[r][1], rg[r][1], 0x2760);                                     // B2 R3 G3 B3
      }
    } else {
      uint32_t px[2][4][3];
#pragma unroll
      for (int jj = 0; jj < 2; jj++) {
        const int j = 2 * q + jj;
        const int c = (int)((cbv[j >> 2] >> (8 * (j & 3))) & 0xffu) - 128, d = (int)((crv[j >> 2] >> (8 * (j & 3))) & 0xffu) - 128;
        const int r_add = K.rv * d + 128, g_add = K.gu * c + K.gv * d + 128, b_add = K.bu * c + 128;
#pragma unroll
        for (int r = 0; r < 2; r++)
#pragma unroll
          for (int i = 0; i < 2; i++) {
            const int p = 2 * jj + i;  // pixel within the group
            const int yy = K.y_mul * ((int)((yv[r][q] >> (8 * p)) & 0xffu) - K.y_sub);
            px[r][p][0] = clip8((yy + r_add) >> 8);
            px[r][p][1] = clip8((yy + g_add) >> 8);
            px[r][p][2] = clip8((yy + b_add) >> 8);
          }
      }
#pragma unroll
      for (int r = 0; r < 2; r++) {
        w[r][3 * q + 0] = pack4(px[r][0][0], px[r][0][1], px[r][0][2], px[r][1][0]);
        w[r][3 * q + 1] = pack4(px[r][1][1], px[r][1][2], px[r][2][0], px[r][2][1]);
        w[r][3 * q + 2] = pack4(px[r][2][2], px[r][3][0], px[r][3][1], px[r][3][2]);
      }
    }
  }
}

template <bool FULL, bool FUSED, bool BULK>
__global__ void __launch_bounds__(kColorThreads) color_stitch_kernel(ColorJob J, Coeffs K, uint32_t row_pairs, uint32_t xblocks) {
  __shared__ __align__(128) uint4 stage[BULK ? 2 * kStageVec : 1];
  const uint32_t per_image = row_pairs * xblocks;
  const uint32_t image = blockIdx.x / per_image, rem = blockIdx.x % per_image;
  const uint32_t y = (rem / xblocks) * 2;
  const uint32_t xb = (rem % xblocks) * kColorThreads * 16;
  const uint32_t x = xb + threadIdx.x * 16;
  const bool in_range = x < J.out_w;  // y < out_h by construction of the grid
  if (!BULK && !in_range) return;
  // tile widths are multiples of 8: the first and the second 8 pixels may lie in different tiles
  const bool two_rows = y + 1 < J.out_h;  // tile heights are even, so row y + 1 is in the same tile
  uint32_t w[2][12];  // packed RGB of the two rows
  if (in_range) convert_block<FULL, FUSED>(J, K, image, x, y, two_rows, w);
  uint8_t* img = J.rgb + (size_t)image * J.image_stride;
  if (BULK) {
    if (in_range) {
#pragma unroll
      for (int r = 0; r < 2; r++) {
        uint4* s = stage + r * kStageVec + threadIdx.x * 3;  // 16-byte stores at a 48-byte stride: conflict-free
        s[0] = make_uint4(w[r][0], w[r][1], w[r][2], w[r][3]);
        s[1] = make_uint4(w[r][4], w[r][5], w[r][6], w[r][7]);
        s[2] = make_uint4(w[r][8], w[r][9], w[r][10], w[r][11]);
      }
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // the writes above, visible to the bulk-copy engine
    __syncthreads();
    if (threadIdx.x == 0) {
      const uint32_t bytes = min(J.out_w - xb, (uint32_t)kColorThreads * 16u) * 3u;  // a multiple of 16 (out_w is one of 16)
      uint8_t* o = img + (size_t)y * J.pitch + (size_t)xb * 3;
      bulk_store(o, stage, bytes);
      if (two_rows) bulk_store(o + J.pitch, stage + kStageVec, bytes);
      asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");  // the staging buffer lives until it has been read
    }
  } else {
#pragma unroll
  for (int r = 0; r < 2; r++) {
    if (r == 1 && !two_rows) break;
    uint8_t* o = img + (size_t)(y + r) * J.pitch + (size_t)x * 3;
    if (x + 16 <= J.out_w && (((uintptr_t)o) & 15u) == 0) {
      reinterpret_cast<uint4*>(o)[0] = make_uint4(w[r][0], w[r][1], w[r][2], w[r][3]);
      reinterpret_cast<uint4*>(o)[1] = make_uint4(w[r][4], w[r][5], w[r][6], w[r][7]);
      reinterpret_cast<uint4*>(o)[2] = make_uint4(w[r][8], w[r][9], w[r][10], w[r][11]);
    } else {
      for (int i = 0; i < 16 && x + i < J.out_w; i++)
        for (int ch = 0; ch < 3; ch++) {
          const int bidx = i * 3 + ch;
          o[bidx] = (uint8_t)(w[r][bidx >> 2] >> (8 * (bidx & 3)));
        }
    }
  }
  }
}

// The 16 x 2 block of convert_block for any geometry, pixel by pixel: any source alignment, blocks that straddle tiles, tiles
// stitched from inside their conformance window (win_x, win_y).  (x, y): canvas position; nx (1..16) pixels of ny (1..2)
// rows are converted, the other bytes are zero.  A pixel's chroma is the sample of its 2x2 quad in the tile's decoded
// picture.  The arithmetic is convert_block's general form (with y_mul = 256, y_sub = 0 it equals the FULL form).
template <bool FUSED>
__device__ __forceinline__ void gather_block(const ColorJob& J, const ColorWindow& G, const Coeffs& K, uint32_t image, uint32_t x,
                                             uint32_t y, uint32_t nx, uint32_t ny, uint32_t (&w)[2][12]) {
#pragma unroll
  for (int r = 0; r < 2; r++) {
#pragma unroll
    for (int q = 0; q < 12; q++) w[r][q] = 0u;
    if ((uint32_t)r >= ny) continue;
    const uint32_t tr = (y + r) / J.tile_h, ly = y + r - tr * J.tile_h + G.win_y;
    uint32_t tc = x / J.tile_w, lx = x - tc * J.tile_w;  // column inside the tile's window
#pragma unroll
    for (int i = 0; i < 16; i++) {
      if ((uint32_t)i < nx) {
        const uint32_t ti = image * J.grid_cols * J.grid_rows + tr * J.grid_cols + tc, sx = lx + G.win_x;
        const uint8_t* t = J.planes + (size_t)ti * J.tile_stride;
        const uint8_t *ty = t, *tcb = t, *tcr = t;
        if (FUSED) {  // as in convert_block; the CTB is found in decoded-picture coordinates
          const uint4 sp = *reinterpret_cast<const uint4*>(J.sao + (size_t)ti * J.sao_stride +
                                                           (size_t)((ly >> J.log2_ctb) * J.wctb + (sx >> J.log2_ctb)) * 4);
          const uint8_t* t2 = J.planes_sao + (size_t)ti * J.tile_stride;
          if (sp.x & 3u) ty = t2;
          if (sp.y & 3u) tcb = t2;
          if (sp.z & 3u) tcr = t2;
        }
        int c = 0, d = 0;
        if (J.chroma) {
          const size_t co = (size_t)(ly >> 1) * J.pitch_c + (sx >> 1);
          c = (int)tcb[J.cb_off + co] - 128;
          d = (int)tcr[J.cr_off + co] - 128;
        }
        const int yy = K.y_mul * ((int)ty[(size_t)ly * J.pitch_y + sx] - K.y_sub);
        const uint32_t px[3] = {clip8((yy + K.rv * d + 128) >> 8), clip8((yy + K.gu * c + K.gv * d + 128) >> 8),
                                clip8((yy + K.bu * c + 128) >> 8)};
#pragma unroll
        for (int ch = 0; ch < 3; ch++) w[r][(3 * i + ch) >> 2] |= px[ch] << (8 * ((3 * i + ch) & 3));
        if (++lx == J.tile_w) lx = 0, tc++;
      }
    }
  }
}

// Everything color_stitch_kernel does not take: a crop at any offset, any of the 8 orientations of heic_image_transform,
// tiles stitched from inside a conformance window or at widths that are not multiples of 8.  A CTA converts a 64 x 64 block
// of the crop rectangle and lays it down in shared memory in output orientation, so that the rows of the output leave as
// contiguous runs of 16-byte stores (a per-pixel scatter to HBM wrote 3 bytes per store).  Crop position (sx, sy) of a
// W x H crop -> output (dx, dy), for the quarter turns:
//   1: (sy, W - 1 - sx)    2: (W - 1 - sx, H - 1 - sy)    3: (H - 1 - sy, sx)
// and then dx -> (output width) - 1 - dx when the mirror bit is set.
// aligned: no window offset, crop origin at x % 8 == 0 and y % 2 == 0, stitch seams at multiples of 8 columns and 2 rows,
// so convert_block's 8-pixel loads apply; otherwise gather_block.
constexpr int kRotTile = 64;
constexpr int kRotRowBytes = kRotTile * 3 + 16;  // padded row of the oriented block (a multiple of 16)

template <bool FULL, bool FUSED>
__global__ void __launch_bounds__(kColorThreads) color_geom_kernel(ColorJob J, ColorWindow G, Coeffs K, uint32_t tiles_x, uint32_t tiles_y,
                                                                   uint32_t aligned) {
  __shared__ __align__(16) uint8_t tile[kRotTile * kRotRowBytes];
  const uint32_t per_image = tiles_x * tiles_y;
  const uint32_t image = blockIdx.x / per_image, rem = blockIdx.x % per_image;
  const uint32_t x0 = (rem % tiles_x) * kRotTile, y0 = (rem / tiles_x) * kRotTile;  // block origin in the crop
  const uint32_t w_v = min((uint32_t)kRotTile, G.crop_w - x0), h_v = min((uint32_t)kRotTile, G.crop_h - y0);  // valid part
  // a warp takes a 16-pixel column strip of the block, a lane two of its rows
  const uint32_t lx = (threadIdx.x >> 5) * 16, ly = (threadIdx.x & 31) * 2;
  const uint32_t rot = J.orientation & 3u;
  const bool mir = (J.orientation & 4u) != 0;
  const uint32_t n_cols = (rot & 1u) ? h_v : w_v, n_rows = (rot & 1u) ? w_v : h_v;  // the block in output orientation
  if (lx < w_v && ly < h_v) {
    const bool two_rows = ly + 1 < h_v;
    const uint32_t cx = G.crop_x + x0 + lx, cy = G.crop_y + y0 + ly;
    uint32_t w[2][12];
    if (aligned) convert_block<FULL, FUSED>(J, K, image, cx, cy, cy + 1 < J.out_h, w);
    else gather_block<FUSED>(J, G, K, image, cx, cy, min(16u, w_v - lx), two_rows ? 2u : 1u, w);
    // byte b (0..47) of row r's 48 bytes of RGB
#define HEIC_RGB_BYTE(r, b) ((w[r][(b) >> 2] >> (8 * ((b) & 3))) & 0xffu)
    // two such bytes as one 16-bit value (low byte first): one PRMT
#define HEIC_RGB_PAIR(ra, ba, rb, bb) __byte_perm(w[ra][(ba) >> 2], w[rb][(bb) >> 2], ((ba) & 3) | ((4 + ((bb) & 3)) << 4))
    if ((rot & 1u) && two_rows && lx + 16 <= w_v && !(h_v & 1u)) {
      // odd quarter turns: the two rows of a column are two neighbouring pixels of one output row -- six contiguous bytes
      // at an even address, written as three 16-bit stores, the upper canvas row first for turn 1 and for turn 3 mirrored
      const bool upper_first = (rot == 1u) != mir;
      const uint32_t col = upper_first ? ly : h_v - 2 - ly;
#pragma unroll
      for (int i = 0; i < 16; i++) {
        const uint32_t sx = lx + i;
        uint16_t* o16 = reinterpret_cast<uint16_t*>(tile + (rot == 1u ? w_v - 1 - sx : sx) * kRotRowBytes + col * 3);
        if (upper_first) {
          o16[0] = (uint16_t)HEIC_RGB_PAIR(0, 3 * i, 0, 3 * i + 1);
          o16[1] = (uint16_t)HEIC_RGB_PAIR(0, 3 * i + 2, 1, 3 * i);
          o16[2] = (uint16_t)HEIC_RGB_PAIR(1, 3 * i + 1, 1, 3 * i + 2);
        } else {
          o16[0] = (uint16_t)HEIC_RGB_PAIR(1, 3 * i, 1, 3 * i + 1);
          o16[1] = (uint16_t)HEIC_RGB_PAIR(1, 3 * i + 2, 0, 3 * i);
          o16[2] = (uint16_t)HEIC_RGB_PAIR(0, 3 * i + 1, 0, 3 * i + 2);
        }
      }
    } else if (((rot == 0 && !mir) || (rot == 2 && mir)) && lx + 16 <= w_v) {
      // unturned, or flipped top <-> bottom: the thread's 48 bytes of each row stay contiguous and in order (and 16-byte
      // aligned: lx * 3 is a multiple of 48)
#pragma unroll
      for (int r = 0; r < 2; r++) {
        if (r == 1 && !two_rows) break;
        uint4* s = reinterpret_cast<uint4*>(tile + (rot == 0 ? ly + r : h_v - 1 - ly - r) * kRotRowBytes + lx * 3);
        s[0] = make_uint4(w[r][0], w[r][1], w[r][2], w[r][3]);
        s[1] = make_uint4(w[r][4], w[r][5], w[r][6], w[r][7]);
        s[2] = make_uint4(w[r][8], w[r][9], w[r][10], w[r][11]);
      }
    } else {
#pragma unroll
      for (int r = 0; r < 2; r++) {
        if (r == 1 && !two_rows) break;
        const uint32_t sy = ly + r;
#pragma unroll
        for (int i = 0; i < 16; i++) {
          const uint32_t sx = lx + i;
          if (sx < w_v) {
            uint32_t row, col;  // position inside the oriented block
            if (rot == 0) row = sy, col = sx;
            else if (rot == 1) row = w_v - 1 - sx, col = sy;
            else if (rot == 2) row = h_v - 1 - sy, col = w_v - 1 - sx;
            else row = sx, col = h_v - 1 - sy;
            if (mir) col = n_cols - 1 - col;
            uint8_t* o = tile + row * kRotRowBytes + col * 3;
            o[0] = (uint8_t)HEIC_RGB_BYTE(r, 3 * i);
            o[1] = (uint8_t)HEIC_RGB_BYTE(r, 3 * i + 1);
            o[2] = (uint8_t)HEIC_RGB_BYTE(r, 3 * i + 2);
          }
        }
      }
    }
#undef HEIC_RGB_BYTE
#undef HEIC_RGB_PAIR
  }
  __syncthreads();
  // oriented block -> HBM
  const uint32_t W = G.crop_w, H = G.crop_h;
  uint32_t dx0, dy0;
  if (rot == 0) dx0 = x0, dy0 = y0;
  else if (rot == 1) dx0 = y0, dy0 = W - x0 - w_v;
  else if (rot == 2) dx0 = W - x0 - w_v, dy0 = H - y0 - h_v;
  else dx0 = H - y0 - h_v, dy0 = x0;
  if (mir) dx0 = ((rot & 1u) ? H : W) - dx0 - n_cols;
  uint8_t* dst = J.rgb + (size_t)image * J.image_stride + (size_t)dy0 * J.pitch + (size_t)dx0 * 3;
  const uint32_t row_bytes = n_cols * 3;
  if (((row_bytes | (uint32_t)J.pitch | (uint32_t)((uintptr_t)dst)) & 15u) == 0) {
    const uint32_t chunks = row_bytes >> 4;
    for (uint32_t q = threadIdx.x; q < n_rows * chunks; q += kColorThreads) {
      const uint32_t row = q / chunks, c = q - row * chunks;
      *reinterpret_cast<uint4*>(dst + (size_t)row * J.pitch + c * 16) = *reinterpret_cast<const uint4*>(tile + row * kRotRowBytes + c * 16);
    }
  } else {
    for (uint32_t q = threadIdx.x; q < n_rows * row_bytes; q += kColorThreads) {
      const uint32_t row = q / row_bytes, c = q - row * row_bytes;
      dst[(size_t)row * J.pitch + c] = tile[row * kRotRowBytes + c];
    }
  }
}

// Box reduction by k = 2..16 fused into the colour pass: the output is PIL.Image.reduce(k) of the RGB color_geom_kernel
// writes, i.e. of T = the crop turned and mirrored.  Output pixel = block of n = rows x cols pixels of T (k x k, fewer in
// its last row and column) with channel sums S, out = (((S + n / 2) * M(n)) mod 2^32) >> 24, M(n) = trunc(float32(2^32) /
// float32(256 n)) (Pillow's fixed-point division, not the rounded mean).
// The sums are taken in crop order and each finished block is placed at its oriented position: along a crop axis that
// the orientation reverses, T's block grid starts at the crop's high edge, so block b covers crop positions
// [b k - p, b k - p + k) with the phase p = (k - L % k) % k on that axis (0 on the others), and the grid of blocks is
// oriented like the grid of pixels.
// A CTA takes a region of kReduceRegionW x kReduceRegionH crop pixels rounded down to whole blocks.  Its threads convert
// crop-aligned 16 x 2 groups (convert_block or gather_block, as color_geom_kernel), add each run of pixels of one block
// in registers -- R + (G << 16) and B: a block sum is at most 256 x 255 < 2^16 -- and add the run into shared memory; then
// the finished pixels are laid down in output orientation and leave as 16-byte stores.
struct ReduceGeom {
  uint32_t k, px, py;        // factor; phase of the block grid along crop x / y
  uint32_t nbx, nby;         // blocks across / down the crop: ceil(crop_w / k), ceil(crop_h / k)
  uint32_t bw, bh;           // blocks of a CTA's region
  uint32_t regions_x, regions_y;
};
constexpr int kReduceRegionW = 256, kReduceRegionH = 32;
constexpr int kReduceBlocks = (kReduceRegionW / 2) * (kReduceRegionH / 2);
constexpr int kReduceSums = kReduceBlocks + kReduceBlocks / 32;  // block i at i + i / 32: a warp's adds hit distinct banks
// the oriented region, rows padded to 16 bytes plus the destination's offset in its 16 bytes: at most 8192 bytes
// (k = 2, odd quarter turn: 128 rows of up(15 + 16 x 3, 16))
constexpr int kReduceStage = 8192;

__device__ __forceinline__ uint32_t reduce_slot(uint32_t i) { return i + (i >> 5); }

// Adds pixels i0..i1-1 of the group's rows in `rows` (bit r: row r) into consecutive blocks from slot `idx`; pixel i0 is
// pixel `c` of its block.
__device__ __forceinline__ void reduce_run(const uint32_t (&w)[2][12], uint32_t rows, uint32_t i0, uint32_t i1, uint32_t c,
                                           uint32_t k, uint32_t idx, uint32_t* sum_rg, uint32_t* sum_b) {
  uint32_t rg = 0, b = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) {
    if ((uint32_t)i < i0 || (uint32_t)i >= i1) continue;
#pragma unroll
    for (int r = 0; r < 2; r++) {
      if (!((rows >> r) & 1u)) continue;
      // R to byte 0 and G to byte 2 (from the one or two words holding them), B alone
      rg += __byte_perm(w[r][(3 * i) >> 2], w[r][(3 * i + 1) >> 2], ((3 * i) & 3) | ((4 + ((3 * i + 1) & 3)) << 8)) & 0x00ff00ffu;
      b += __byte_perm(w[r][(3 * i + 2) >> 2], 0u, 0x4440 | ((3 * i + 2) & 3));
    }
    if (++c == k || (uint32_t)i + 1 == i1) {
      atomicAdd(sum_rg + reduce_slot(idx), rg);
      atomicAdd(sum_b + reduce_slot(idx), b);
      rg = b = 0;
      c = 0;
      idx++;
    }
  }
}

template <bool FULL, bool FUSED>
__global__ void __launch_bounds__(kColorThreads) color_reduce_kernel(ColorJob J, ColorWindow G, Coeffs K, ReduceGeom R, uint32_t aligned) {
  __shared__ uint32_t sum_rg[kReduceSums], sum_b[kReduceSums];
  __shared__ __align__(16) uint8_t stage[kReduceStage];
  const uint32_t per_image = R.regions_x * R.regions_y;
  const uint32_t image = blockIdx.x / per_image, rem = blockIdx.x % per_image;
  const uint32_t bx0 = (rem % R.regions_x) * R.bw, by0 = (rem / R.regions_x) * R.bh;  // first block of the region
  const uint32_t bw = min(R.bw, R.nbx - bx0), bh = min(R.bh, R.nby - by0);
  const int k = (int)R.k, W = (int)G.crop_w, H = (int)G.crop_h;
  const uint32_t n_slots = reduce_slot(R.bw * bh - 1) + 1;
  for (uint32_t i = threadIdx.x; i < n_slots; i += kColorThreads) sum_rg[i] = sum_b[i] = 0u;
  // the region's pixels in crop coordinates, and the crop-aligned 16 x 2 groups that cover them
  const int xs = max(0, (int)bx0 * k - (int)R.px), xe = min(W, (int)(bx0 + bw) * k - (int)R.px);
  const int ys = max(0, (int)by0 * k - (int)R.py), ye = min(H, (int)(by0 + bh) * k - (int)R.py);
  const uint32_t gx0 = (uint32_t)xs / 16, gy0 = (uint32_t)ys / 2;
  const uint32_t ngx = (uint32_t)(xe - 1) / 16 - gx0 + 1, ngy = (uint32_t)(ye - 1) / 2 - gy0 + 1;
  __syncthreads();
  for (uint32_t g = threadIdx.x; g < ngx * ngy; g += kColorThreads) {
    const int sx0 = (int)(gx0 + g % ngx) * 16, sy0 = (int)(gy0 + g / ngx) * 2;
    const uint32_t cx = G.crop_x + (uint32_t)sx0, cy = G.crop_y + (uint32_t)sy0;
    uint32_t w[2][12];
    if (aligned) convert_block<FULL, FUSED>(J, K, image, cx, cy, cy + 1 < J.out_h, w);
    else gather_block<FUSED>(J, G, K, image, cx, cy, (uint32_t)min(16, W - sx0), sy0 + 1 < H ? 2u : 1u, w);
    const int x_first = max(xs, sx0);
    const uint32_t i0 = (uint32_t)(x_first - sx0), i1 = (uint32_t)(min(xe, sx0 + 16) - sx0);
    const uint32_t c = (uint32_t)(x_first + (int)R.px) % (uint32_t)k;
    const uint32_t lbx = (uint32_t)(x_first + (int)R.px) / (uint32_t)k - bx0;
    const bool r0 = sy0 >= ys, r1 = sy0 + 1 < ye;  // rows of the group inside the region
    const uint32_t lby0 = (uint32_t)(sy0 + (int)R.py) / (uint32_t)k - by0, lby1 = (uint32_t)(sy0 + 1 + (int)R.py) / (uint32_t)k - by0;
    if (r0 && r1 && lby0 == lby1) {
      reduce_run(w, 3u, i0, i1, c, (uint32_t)k, lby0 * R.bw + lbx, sum_rg, sum_b);
    } else {
      if (r0) reduce_run(w, 1u, i0, i1, c, (uint32_t)k, lby0 * R.bw + lbx, sum_rg, sum_b);
      if (r1) reduce_run(w, 2u, i0, i1, c, (uint32_t)k, lby1 * R.bw + lbx, sum_rg, sum_b);
    }
  }
  __syncthreads();
  // the region in output orientation: the block grid is oriented as color_geom_kernel orients the pixel grid
  const uint32_t rot = J.orientation & 3u;
  const bool mir = (J.orientation & 4u) != 0;
  const uint32_t n_cols = (rot & 1u) ? bh : bw, n_rows = (rot & 1u) ? bw : bh;
  uint32_t dx0, dy0;
  if (rot == 0) dx0 = bx0, dy0 = by0;
  else if (rot == 1) dx0 = by0, dy0 = R.nbx - bx0 - bw;
  else if (rot == 2) dx0 = R.nbx - bx0 - bw, dy0 = R.nby - by0 - bh;
  else dx0 = R.nby - by0 - bh, dy0 = bx0;
  if (mir) dx0 = ((rot & 1u) ? R.nby : R.nbx) - dx0 - n_cols;
  uint8_t* dst = J.rgb + (size_t)image * J.image_stride + (size_t)dy0 * J.pitch + (size_t)dx0 * 3;
  // staging rows start at the destination's offset inside its 16 bytes, so that whole 16-byte words go out as one store
  const bool wide = ((J.pitch | J.image_stride | (uint64_t)(uintptr_t)J.rgb) & 15u) == 0;
  const uint32_t a = wide ? (uint32_t)((uintptr_t)dst & 15u) : 0u;
  const uint32_t row_bytes = n_cols * 3, rs = (a + row_bytes + 15u) & ~15u;
  for (uint32_t t = threadIdx.x; t < bw * bh; t += kColorThreads) {
    const uint32_t lbx = t % bw, lby = t / bw;
    const int x0 = (int)(bx0 + lbx) * k - (int)R.px, y0 = (int)(by0 + lby) * k - (int)R.py;
    const uint32_t n = (uint32_t)((min(x0 + k, W) - max(x0, 0)) * (min(y0 + k, H) - max(y0, 0)));
    const uint32_t m = __float2uint_rz(__fdiv_rn(4294967296.0f, (float)(256u * n))), half = n >> 1;
    const uint32_t s = reduce_slot(lby * R.bw + lbx), rg = sum_rg[s], b = sum_b[s];
    uint32_t row, col;
    if (rot == 0) row = lby, col = lbx;
    else if (rot == 1) row = bw - 1 - lbx, col = lby;
    else if (rot == 2) row = bh - 1 - lby, col = bw - 1 - lbx;
    else row = lbx, col = bh - 1 - lby;
    if (mir) col = n_cols - 1 - col;
    uint8_t* o = stage + row * rs + a + col * 3;
    o[0] = (uint8_t)((((rg & 0xffffu) + half) * m) >> 24);
    o[1] = (uint8_t)((((rg >> 16) + half) * m) >> 24);
    o[2] = (uint8_t)(((b + half) * m) >> 24);
  }
  __syncthreads();
  if (wide) {
    uint8_t* base = dst - a;  // 16-byte aligned; the row's bytes are [a, a + row_bytes) of each staging row
    const uint32_t chunks = rs >> 4;
    for (uint32_t q = threadIdx.x; q < n_rows * chunks; q += kColorThreads) {
      const uint32_t row = q / chunks, b0 = (q - row * chunks) * 16;
      uint8_t* d = base + (size_t)row * J.pitch;
      const uint8_t* s = stage + row * rs;
      if (b0 >= a && b0 + 16 <= a + row_bytes) {
        *reinterpret_cast<uint4*>(d + b0) = *reinterpret_cast<const uint4*>(s + b0);
      } else {  // the row's partial first and last 16 bytes: the neighbouring regions write the rest
        for (uint32_t j = max(b0, a); j < min(b0 + 16, a + row_bytes); j++) d[j] = s[j];
      }
    }
  } else {
    for (uint32_t q = threadIdx.x; q < n_rows * row_bytes; q += kColorThreads) {
      const uint32_t row = q / row_bytes, c = q - row * row_bytes;
      dst[(size_t)row * J.pitch + c] = stage[row * rs + c];
    }
  }
}

}  // namespace

cudaError_t launch_color(const ColorJob& job, const ColorWindow& win, uint32_t reduce, cudaStream_t stream) {
  if (!job.n_images || !job.out_w || !job.out_h || !win.crop_w || !win.crop_h) return cudaSuccess;
  Coeffs k;
  const bool bt709 = job.matrix_coeffs == 1;
  if (job.full_range) {
    k.y_mul = 256;
    k.y_sub = 0;
    if (bt709) k.rv = 403, k.gu = -48, k.gv = -120, k.bu = 475;
    else k.rv = 359, k.gu = -88, k.gv = -183, k.bu = 454;
  } else {
    k.y_mul = 298;
    k.y_sub = 16;
    if (bt709) k.rv = 459, k.gu = -55, k.gv = -136, k.bu = 541;
    else k.rv = 409, k.gu = -100, k.gv = -208, k.bu = 516;
  }
  // seams between tiles at multiples of 8 columns and of 2 rows (or none): the first and the second 8 pixels of a
  // 16-pixel group may lie in different tiles, not within one, and the two rows of a thread lie in one tile
  const bool seams = (job.tile_w % 8 == 0 || job.grid_cols == 1) && (job.tile_h % 2 == 0 || job.grid_rows == 1);
  if (reduce > 1) {
    const uint32_t rot = job.orientation & 3u;
    const bool mir = (job.orientation & 4u) != 0;
    // crop axes that the orientation reverses (see color_reduce_kernel)
    const bool rev_x = rot == 1 || (rot == 0 && mir) || (rot == 2 && !mir), rev_y = rot == 2 || (rot == 1 && mir) || (rot == 3 && !mir);
    ReduceGeom r;
    r.k = reduce;
    r.px = rev_x ? (reduce - win.crop_w % reduce) % reduce : 0u;
    r.py = rev_y ? (reduce - win.crop_h % reduce) % reduce : 0u;
    r.nbx = (win.crop_w + reduce - 1) / reduce;
    r.nby = (win.crop_h + reduce - 1) / reduce;
    r.bw = (uint32_t)kReduceRegionW / reduce;  // k <= 16: at least 16 x 2 blocks
    r.bh = (uint32_t)kReduceRegionH / reduce;
    r.regions_x = (r.nbx + r.bw - 1) / r.bw;
    r.regions_y = (r.nby + r.bh - 1) / r.bh;
    const unsigned grid = job.n_images * r.regions_x * r.regions_y;
    const uint32_t aligned = !win.win_x && !win.win_y && seams && win.crop_x % 8 == 0 && win.crop_y % 2 == 0;
    if (job.fused) {
      if (job.full_range) color_reduce_kernel<true, true><<<grid, kColorThreads, 0, stream>>>(job, win, k, r, aligned);
      else color_reduce_kernel<false, true><<<grid, kColorThreads, 0, stream>>>(job, win, k, r, aligned);
    } else {
      if (job.full_range) color_reduce_kernel<true, false><<<grid, kColorThreads, 0, stream>>>(job, win, k, r, aligned);
      else color_reduce_kernel<false, false><<<grid, kColorThreads, 0, stream>>>(job, win, k, r, aligned);
    }
    return cudaGetLastError();
  }
  if (job.orientation != 0 || win.crop_x || win.crop_y || win.win_x || win.win_y || !seams) {
    const uint32_t tiles_x = (win.crop_w + kRotTile - 1) / kRotTile, tiles_y = (win.crop_h + kRotTile - 1) / kRotTile;
    const unsigned rgrid = job.n_images * tiles_x * tiles_y;
    const uint32_t aligned = !win.win_x && !win.win_y && seams && win.crop_x % 8 == 0 && win.crop_y % 2 == 0;
    if (job.fused) {
      if (job.full_range) color_geom_kernel<true, true><<<rgrid, kColorThreads, 0, stream>>>(job, win, k, tiles_x, tiles_y, aligned);
      else color_geom_kernel<false, true><<<rgrid, kColorThreads, 0, stream>>>(job, win, k, tiles_x, tiles_y, aligned);
    } else {
      if (job.full_range) color_geom_kernel<true, false><<<rgrid, kColorThreads, 0, stream>>>(job, win, k, tiles_x, tiles_y, aligned);
      else color_geom_kernel<false, false><<<rgrid, kColorThreads, 0, stream>>>(job, win, k, tiles_x, tiles_y, aligned);
    }
    return cudaGetLastError();
  }
  // the crop is a top-left part of the canvas: the stitch kernel, with the crop as its canvas
  ColorJob j = job;
  j.out_w = win.crop_w;
  j.out_h = win.crop_h;
  const uint32_t groups = (j.out_w + 15) / 16;
  const uint32_t xblocks = (groups + kColorThreads - 1) / kColorThreads, row_pairs = (j.out_h + 1) / 2;
  const unsigned grid = j.n_images * row_pairs * xblocks;
  // bulk (TMA) stores need 16-byte aligned rows whose length is a multiple of 16 bytes
  const bool bulk = j.out_w % 16 == 0 && j.pitch % 16 == 0 && j.image_stride % 16 == 0 && ((uintptr_t)j.rgb & 15u) == 0;
#define HEIC_COLOR_LAUNCH(FULL, FUSED)                                                                                  \
  do {                                                                                                                  \
    if (bulk) color_stitch_kernel<FULL, FUSED, true><<<grid, kColorThreads, 0, stream>>>(j, k, row_pairs, xblocks);     \
    else color_stitch_kernel<FULL, FUSED, false><<<grid, kColorThreads, 0, stream>>>(j, k, row_pairs, xblocks);         \
  } while (0)
  if (job.fused) {
    if (job.full_range) HEIC_COLOR_LAUNCH(true, true);
    else HEIC_COLOR_LAUNCH(false, true);
  } else {
    if (job.full_range) HEIC_COLOR_LAUNCH(true, false);
    else HEIC_COLOR_LAUNCH(false, false);
  }
#undef HEIC_COLOR_LAUNCH
  return cudaGetLastError();
}

}  // namespace dev
}  // namespace heic
