// Launchers of the sm_100a kernels (one translation unit per stage).
#pragma once
#include <cuda_runtime.h>

#include "dev_types.h"

namespace heic {
namespace dev {

struct CabacTabs;

// Stage 1 — CABAC: slice data -> tu_map / TransCoeffLevel / QpY / SAO parameters.
// order: n_groups * tiles_per_cta tile indices (0xffffffff = idle lane); all tiles of one group share
// their PicParams geometry.  n_slots = row slots (warps) per CTA.
size_t cabac_smem_bytes(int tiles_per_cta, int n_slots);
// group_counter: a zeroed device word; when given (and there is more than one wave of groups) the thread-per-substream
// mapping runs as persistent CTAs that take their groups from it
cudaError_t launch_cabac(const Arenas& A, const CabacTabs* tabs, const uint32_t* order, uint32_t n_groups,
                         int tiles_per_cta, int n_slots, uint32_t* group_counter, int n_sm, int resident_ctas /* 0: fill the GPU */,
                         cudaStream_t stream);

// Stage 2 — scaling (8.6.4.2) + inverse DST/DCT (8.6.4.2), in place on the coefficient arena.
// Emulation-prevention removal (7.4.2 / rbsp_reader.rs:11-39) and entry-point re-basing for the tiles shipped raw:
// raw arena -> bitstream arena, and bs_len / data_off / substream offsets rewritten in un-escaped bytes.
cudaError_t launch_unescape(const Arenas& A, TileParams* tiles, uint32_t* substreams, cudaStream_t stream);
cudaError_t launch_transform(const Arenas& A, uint32_t max_tu_per_tile, int max_log2_tb, int n_sm, cudaStream_t stream);
// element offsets of the per-class coded-block lists for `total_tu` tu_map entries; returns the total element count
size_t transform_list_layout(size_t total_tu, uint32_t off[LIST_CLASSES]);
int transform_launches(int max_log2_tb);

// Stage 3 — intra prediction + reconstruction (8.4.4.2), CTU wavefront per picture.
// order: every tile index once, heaviest first (launch order of the one-CTA-per-picture grid)
// clear_coeff: zero every coefficient slot after consuming it (leaves the arena ready for the next decode's CABAC stage)
cudaError_t launch_intra(const Arenas& A, const uint32_t* order, int max_log2_ctb, int max_hctb, int n_slots, bool clear_coeff,
                         cudaStream_t stream);

// Stage 4 — deblocking (8.7.2), in place on the reconstruction arena.
cudaError_t launch_deblock(const Arenas& A, uint32_t max_w, uint32_t max_h, cudaStream_t stream);

// Stage 5 — SAO (8.7.3): recon arena -> final arena.
cudaError_t launch_sao(const Arenas& A, uint32_t max_pitch, uint32_t max_h, cudaStream_t stream);
// The same for the CTBs with SAO switched on only (the others are left untouched in the final arena): what a decode to RGB
// runs, followed by a colour kernel that picks every CTB's component from the arena holding its final samples.
cudaError_t launch_sao_sparse(const Arenas& A, int max_hctb, cudaStream_t stream);

// Stage 6 — YCbCr 4:2:0 -> RGB8 + grid stitch + crop (+ orientation).
struct ColorJob {
  const uint8_t* planes;        // tile t: planes + t * tile_stride; Y then Cb then Cr
  uint64_t tile_stride;         // bytes between tiles
  uint64_t cb_off, cr_off;      // offsets of Cb / Cr inside a tile
  uint32_t pitch_y, pitch_c;
  uint32_t tile_w, tile_h;      // size at which the grid stitches a tile (its conformance window)
  uint32_t grid_cols, grid_rows;
  uint32_t out_w, out_h;        // canvas (before the crop and the orientation)
  uint32_t n_images;            // images are consecutive groups of grid_cols*grid_rows tiles
  uint32_t chroma;              // 0: monochrome (Cb = Cr = 128)
  uint32_t full_range, matrix_coeffs;
  uint32_t orientation;         // heic_image_transform::orientation applied to the output
  uint8_t* rgb;
  uint64_t pitch, image_stride; // output layout in bytes
  // fused == 1: `planes` is the deblocked reconstruction, and a CTB component whose SAO type is non-zero is read from
  // `planes_sao` instead (the final arena, same layout, filled for those CTBs by launch_sao_sparse)
  uint32_t fused;
  const uint8_t* planes_sao;
  const uint32_t* sao;          // SAO parameters of the job's first tile (4 words per CTB; all-zero where SAO is off)
  uint32_t sao_stride;          // words between tiles
  uint32_t log2_ctb, wctb;
};
// The rest of the output geometry.  It travels beside ColorJob rather than inside it: the stitch kernel takes ColorJob by
// value, and a longer ColorJob would move the kernel parameters after it.
struct ColorWindow {
  uint32_t crop_x, crop_y, crop_w, crop_h;  // output rectangle in canvas coordinates, before the orientation
  uint32_t win_x, win_y;                    // origin of a tile's stitched part inside its decoded picture (luma samples)
};
// reduce = 1: identity orientation, crop and window at the origin, tiles stitched at multiples of 8 pixels:
// color_stitch_kernel; everything else: color_geom_kernel.
// reduce = 2..16: color_reduce_kernel writes PIL.Image.reduce(reduce) of that output (include/heic_b200.h,
// heic_b200_decode_grids_reduced): ceil(w / reduce) x ceil(h / reduce) pixels.
cudaError_t launch_color(const ColorJob& job, const ColorWindow& win, uint32_t reduce, cudaStream_t stream);

}  // namespace dev
}  // namespace heic
